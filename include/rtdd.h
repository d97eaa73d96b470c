/*
 * rtdd.h -- C ABI of librtdd.so, the B200 (sm_100a) implementation of the
 * RealTimeDepthDiffusion hot path.
 *
 * This is the drop-in boundary: plain C, plain pointers and sizes, explicit
 * context handle, int status returns.  Each entry point names the reference
 * interface it replaces (paths relative to the reference repository).  The
 * reference-named C++ functions of include/GPUSolver.h, GPUImageProcessing.h and
 * GPUDepthEffect.h are thin shims over these (csrc/gpu_shims.cpp) that keep the
 * reference's "void + print + continue" error convention and one process-global
 * context.
 *
 * Unless a parameter says "host", every image pointer is a DEVICE pointer owned
 * by the caller and every pitch is in BYTES, exactly as the reference passes
 * cv::cuda::GpuMat::ptr()/step.  All work is enqueued on the context's stream
 * (rtdd_set_stream; default: a blocking stream, which orders itself against the
 * legacy default stream the way the reference's default-stream launches do).
 *
 * Status: 0 = success; > 0 = a cudaError_t value; < 0 = RTDD_E_* argument/state
 * error.  rtdd_last_error(ctx) returns a printable description of the last
 * non-zero status.  There is no CPU fallback anywhere behind this interface.
 */
#ifndef RTDD_H
#define RTDD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTDD_E_ARG     (-1)   /* bad argument (null pointer, level out of range, size mismatch) */
#define RTDD_E_STATE   (-2)   /* call-order violation (e.g. solve before rtdd_load_weights) */
#define RTDD_E_NOMEM   (-3)   /* host allocation failed */
#define RTDD_E_PEER    (-4)   /* multi-GPU strip set-up failed (no peer access, bad rank layout) */

typedef struct rtdd_ctx rtdd_ctx;

/* ---- life cycle ---------------------------------------------------------- */

/* replaces GPUAllocateDeviceMemory(rows, cols, levels)   ref: include/GPUSolver.h:6, src/GPUSolver.cu:33-54
 * One context per GPU; scratch planes for levels l = 0..levels-1 of size
 * floor(rows/2^l) x floor(cols/2^l) in a single HBM arena.  device < 0 = current device. */
int rtdd_create(int rows, int cols, int levels, int device, rtdd_ctx **out);
/* A context for one rank of a row-strip frame over `nranks` GPUs (rtdd_strip_frame_*): like rtdd_create, but the scratch planes of
 * the levels that get split hold only the largest row window a rank keeps (own rows + `halo` ghost rows per side) instead of the
 * whole level.  Same layout on every rank.  Whole-level calls on such a level return RTDD_E_STATE. */
int rtdd_create_strip(int rows, int cols, int levels, int device, int nranks, int halo, long long minStripPixels, rtdd_ctx **out);
/* replaces GPUFreeDeviceMemory(levels)                    ref: include/GPUSolver.h:7, src/GPUSolver.cu:56-71 */
int rtdd_destroy(rtdd_ctx *ctx);
/* replaces GPULoadWeights(beta)                           ref: include/GPUSolver.h:8, src/GPUSolver.cu:264-272
 * w[i] = expf(-beta * i) for i = 0..255 (host fp32), w[256] = 0.  Deviation: beta < 0 (weights above 1) and NaN or
 * infinite beta (NaN weights) return RTDD_E_ARG and leave the previously loaded table, or none, in force; -0.0 is accepted.
 * The table may be reloaded at any time: later solves, cached graphs included, use the new one. */
int rtdd_load_weights(rtdd_ctx *ctx, float beta);
/* stream = a cudaStream_t (NULL restores the context's own stream). */
int rtdd_set_stream(rtdd_ctx *ctx, void *stream);
/* replaces the cudaThreadSynchronize in GPUCheckError     ref: src/GPUSolver.cu:21-27 */
int rtdd_sync(rtdd_ctx *ctx);
const char *rtdd_last_error(const rtdd_ctx *ctx);
/* number of kernels this context has launched (directly or through graph replays) since creation */
unsigned long long rtdd_launch_count(const rtdd_ctx *ctx);
int rtdd_levels(const rtdd_ctx *ctx);
/* ref: src/main.cpp:95 -- floor(log2(max(min(cols,rows)/45,1)))+1 */
int rtdd_pyramid_levels(int rows, int cols);
/* ref: src/main.cpp:153,263 -- floor(maxIterations / 2^(levels-1-level)) */
int rtdd_level_iterations(int maxIterations, int levels, int level);

/* ---- the solve ----------------------------------------------------------- */

/* replaces GPUMatrixFreeSolver(depth, depthPitch, scribble, scribblePitch, gray, grayPitch,
 *                              rows, cols, beta, maxIterations, tolerance, level)
 * ref: include/GPUSolver.h:9-10, src/GPUSolver.cu:274-316.
 * One pyramid level: edge-weight pass on (gray, incoming depth), maxIterations
 * Chebyshev-Jacobi sweeps with scribble (== 255) Dirichlet masking, result back in
 * `depth` (in place).  beta/tolerance do not exist here because the reference ignores them.
 * Asynchronous on the context stream (the C++ shim adds the reference's device sync). */
int rtdd_solve_level(rtdd_ctx *ctx, float *depth, size_t depthPitch,
                     const uint8_t *scribble, size_t scribblePitch,
                     const uint8_t *gray, size_t grayPitch,
                     int rows, int cols, int maxIterations, int level);

/* The edge-weight pass alone (the reference's file-local loadIndexToWeight kernel,
 * ref: src/GPUSolver.cu:136-224,293), exposed for parity tests and profiling.
 * Writes the packed link indices of `level` into the context and, if the out pointers
 * are non-null, copies them to caller DEVICE planes of pitch outPitch bytes:
 *   linkRight[y][x] = LUT index of the link (x,y)-(x+1,y)   (the reference's `right` of (x,y)
 *                     == `left` of (x+1,y)); 0 in the last column (no such link)
 *   linkDown [y][x] = LUT index of the link (x,y)-(x,y+1);   0 in the last row.
 * Links that leave the image carry weight 0 by position (the reference's index 256). */
int rtdd_edge_weights(rtdd_ctx *ctx, const float *depth, size_t depthPitch,
                      const uint8_t *gray, size_t grayPitch,
                      int rows, int cols, int level,
                      uint8_t *linkRight, uint8_t *linkDown, size_t outPitch);

/* Device time of the sweep kernels of the most recent rtdd_solve_level on `level` (CUDA events on the
 * context stream around the sweep launches; excludes the edge-weight pass and the copy back):
 * the measured counterpart of the reference's per-level `iteration` loop (ref: src/GPUSolver.cu:295-309).
 * Blocks until that work has finished.  iterations/kernels (may be NULL) return the sweep count and
 * the number of kernel launches it took. */
int rtdd_level_sweep_ms(rtdd_ctx *ctx, int level, float *ms, int *iterations, int *kernels);

/* ---- opt-in extensions (NOT the parity path: the reference runs a fixed schedule and never checks convergence,
 *      ref: src/GPUSolver.cu:226,274-275 accept `tolerance` / `deviceError` and never read them) -------------------- */

/* Max-norm of the last sweep's update, max |x_K - x_{K-1}| over the level, of the most recent solve of `level`:
 * a warp-shuffle + atomicMax by-product of the final sweep pass (the slot the reference reserved as deviceError).
 * Blocks until that solve has finished.  *residual is a HOST float. */
int rtdd_level_residual(rtdd_ctx *ctx, int level, float *residual);
/* GPUMatrixFreeSolver with the `tolerance` argument honoured: same sweeps, same omega schedule, but the residual is
 * read back every `checkEvery` sweeps and the level stops early once it is <= tolerance (or at maxIterations).
 * With tolerance = 0 it runs all maxIterations sweeps and equals rtdd_solve_level bit for bit. */
int rtdd_solve_level_converge(rtdd_ctx *ctx, float *depth, size_t depthPitch, const uint8_t *scribble, size_t scribblePitch,
                              const uint8_t *gray, size_t grayPitch, int rows, int cols, int maxIterations, float tolerance,
                              int checkEvery, int level, int *iterationsRun, float *finalResidual);

/* Self-test of the sweep kernels' branch-free division (csrc/solver_kernels.cu: div_fast) against the
 * compiler's IEEE div.rn (the operation the reference's `sum / count` compiles to, ref: src/GPUSolver.cu:104)
 * on n counter-generated operand pairs.  mode 0 = the whole admitted range, 1 = the sweep's typical range,
 * 2 = quotients placed next to rounding boundaries, 3 = tiny/denormal denominators through the exact power-of-two
 * rescaling the resident kernel uses, 4 = numerators below 2^-100 (denormals included) through the resident kernel's
 * exact small-quotient path (div_tiny).  *mismatches (HOST) must come back 0. */
int rtdd_selftest_division(rtdd_ctx *ctx, unsigned long long n, unsigned long long seed, int mode, unsigned long long *mismatches);

/* Sweep implementation selector for rtdd_solve_level: 0 = auto (default),
 * 1 = one sweep per launch, 2 = temporally blocked tiles, 3 = cluster-resident (whole level in the
 * registers of one thread-block cluster for all sweeps; falls back to 2 if the level is too large).  All variants are
 * bit-identical by construction; the selector exists for tests and profiling. */
int rtdd_set_sweep_variant(rtdd_ctx *ctx, int variant, int sweepsPerPass);
/* Process-wide tuning knobs for experiments (tools/tune_blocked.py); results never change, only speed.
 * "blocked_tile": 0 auto, 64 = 128x64-pixel regions, 34 = 128x32 regions with 2 rows per warp, 32 = 128x32 with 4 rows per warp;
 * "blocked_tma": 3 = TMA-fed persistent thread-block clusters (vertically adjacent CTAs share their edge rows over distributed
 *                shared memory), 1 = TMA-fed persistent single CTAs, 2 (default) = clusters for levels >= 2^20 pixels and
 *                single CTAs below (measured), 0 = plain LDG form;
 * "blocked_cluster": CTAs per cluster of the default form (1, 2 (default), 4, 8);
 * "blocked_grid_cap": > 0 limits the persistent form to that many CTAs (tests: every CTA then walks several regions even on
 *                     small levels, so the region loop -- phase flips, re-issue under the sweeps -- is checked against the oracle);
 * "spin_timeout_ms": device-time limit of a halo wait on a neighbouring rank (default 20000, 0 = for ever); a wait that gives
 *                    up marks the context and the next rtdd_sync returns RTDD_E_PEER instead of the context dying;
 * "resident_warps": target warps per CTA of the cluster-resident kernel (default 8);
 * "pdl": 1 (default) sweep passes are chained with programmatic dependent launch, 0 = plain stream order;
 * "strip_residual": 1 = rtdd_strip_pass also fills the level's residual word (rtdd_level_residual), default 0;
 * "strip_peer_staging": 1 = halo rows of a strip level travel through rtdd_strip_push / rtdd_strip_pull, default 0;
 * "fused_prolong": 1 = whole-frame path forms a level's guess inside its set-up kernel, default 0 (no faster, see DESIGN.md);
 * "resident_r1_max_warps": largest one-row-per-warp CTA of the cluster-resident kernel (default 32);
 * "pass_planner": 1 (default) = passes of their own lengths and halos (rtdd_plan_passes), 0 = one length per level (rtdd_plan_blocked);
 * "plan_throughput": per CONTEXT, 1 = its pass plans minimise total SM time instead of the level's latency -- for contexts that keep
 *                    the GPU busy together (several images in flight, rtdd_mgpu_batch_solve sets it on its own contexts), default 0;
 * "zero_copy_out": 1 (default) = rtdd_frame_solve_host* let the last level-0 pass store the 8-bit map straight into the caller's
 *                  plane when that is pinned host memory (4-byte aligned base and pitch) and level 0 runs at least 8 sweeps,
 *                  0 = always the staged copy. */
int rtdd_set_tuning(rtdd_ctx *ctx, const char *key, int value);

/* ---- row strips: one level of one very large image split across GPUs (BASELINE configs[4]) --------
 * No reference counterpart (the reference is single-GPU); results are bit-identical to rtdd_solve_level.
 * A rank keeps rows [winBegin, winEnd) of the level = its own rows plus H ghost rows on each side that is not an
 * image edge.  rtdd_strip_init = the edge-weight pass on the window (ref: src/GPUSolver.cu:290-293);
 * rtdd_strip_pass = nsweeps (<= haloT <= H) sweeps starting at sweep index firstSweep of the level's schedule
 * (ref: src/GPUSolver.cu:295-309); afterwards the nsweeps rows next to a non-image window edge are stale and
 * must be refreshed from the neighbouring rank before the next pass: rtdd_strip_planes returns the device
 * planes holding x_k and x_{k-1} (row 0 = winBegin, row pitch pitchBytes) to send from / receive into;
 * rtdd_strip_finish copies final rows [rowBegin, rowEnd) (level coordinates) into the pitched depth plane. */
/* Host-side planning of the decomposition (no device work).  rtdd_plan_strips: levels are finest first; for every split
 * level l, split[l] = 1 and rank r owns rows [ownBegin[l * nranks + r], ownEnd[l * nranks + r]); the coarsest split level
 * is cut evenly and every finer one doubles its boundaries.  rtdd_strip_schedule: the passes of one split level and the
 * halo exchanges between them (several passes of passSweeps <= halo sweeps may share one exchange); returns the number
 * of passes, negative on error. */
int rtdd_plan_strips(const int *levelRows, const int *levelCols, int levels, int nranks, int halo, long long minStripPixels,
                     int *split, int *ownBegin, int *ownEnd);
int rtdd_strip_schedule(int iters, int halo, int passSweeps, int level, int *sweepsOfPass, int *exchangeAfter, int capacity);
/* host only: planeRows[l] = rows the scratch planes of level l hold on every rank of a strip frame (rtdd_create_strip) */
int rtdd_plan_strip_planes(const int *levelRows, const int *levelCols, int levels, int nranks, int halo, long long minStripPixels, int *planeRows);
/* host only: how rtdd_solve_level runs `iterations` sweeps of a rows x cols level (>= 2^18 pixels) with the temporally blocked
 * kernels on a GPU of smCount SMs: sweeps per pass (= per HBM round trip) and whether thread-block clusters of two CTAs sweep
 * 128 x 128 regions (1) or single CTAs 128 x 64 ones (0).  A cost model fitted to measurements (DESIGN.md section 3). */
int rtdd_plan_blocked(int rows, int cols, int iterations, int smCount, int *sweepsPerPass, int *clusterForm);
/* host only: the passes the level driver actually runs (default; rtdd_set_tuning("pass_planner", 0) returns to one length per
 * level): the same cost model, every pass with the halo of its own length, lengths chosen by a small dynamic programme
 * (3840 x 2160 x 31 sweeps: 7, 7, 7, 10).  flags & 1: the last pass also stores the 8-bit map into pinned host memory
 * (rtdd_frame_solve_host*) and is made as long as the tiling allows, so that the transfer hides under its sweeps (7, 8, 16);
 * flags & 2: the plan of a context that shares the GPU with others (rtdd_set_tuning "plan_throughput"): least total SM time
 * instead of least latency.  *clusterForm: 1 = clusters of two CTAs on 128 x 128 regions, 0 = single CTAs on 128 x 64 regions,
 * 2 = single CTAs on 128 x 32 regions (levels below 2^18 pixels only).  Returns the number of passes (the last pass last),
 * negative on error. */
int rtdd_plan_passes(int rows, int cols, int iterations, int smCount, int flags, int *sweepsOfPass, int capacity, int *clusterForm);
/* The caller's own pass lengths (1..16 sweeps each) for one level of the temporally blocked kernels -- tuning and tests; used
 * whenever the level is solved with exactly their total, npasses = 0 removes them.  Results do not depend on the plan. */
int rtdd_set_pass_plan(rtdd_ctx *ctx, int level, const int *sweepsOfPass, int npasses);
int rtdd_strip_init(rtdd_ctx *ctx, int level, const float *depth, size_t depthPitch, const uint8_t *scribble, size_t scribblePitch,
                    const uint8_t *gray, size_t grayPitch, int rows, int cols, int winBegin, int winEnd);
int rtdd_strip_pass(rtdd_ctx *ctx, int level, int firstSweep, int nsweeps, int haloT);
int rtdd_strip_planes(rtdd_ctx *ctx, int level, float **xk, float **xkm1, size_t *pitchBytes, int *winBegin, int *winRows);
int rtdd_strip_finish(rtdd_ctx *ctx, int level, float *depth, size_t depthPitch, int rowBegin, int rowEnd);
/* Fused halo exchange: instead of handing the halo rows to NCCL, the sweep pass itself stores the rows next to a strip
 * boundary into the neighbouring rank's ghost rows (peer memory, NVLink) and raises a flag there; the neighbour's
 * next pass waits for that flag on the device.  Every rank's arena has the same layout, so a neighbour is described
 * by the base of its arena: rtdd_ipc_export / rtdd_ipc_import move a CUDA IPC handle (64 bytes) between processes
 * (rtdd_arena gives the base directly for contexts of one process).  rtdd_strip_neighbours, called after
 * rtdd_strip_init, gives this rank's own rows [ownBegin, ownEnd), the halo depth and the first row of the windows of
 * the ranks above / below (-1 = none) and switches the level to the fused mode; rtdd_strip_wait enqueues the wait for
 * the neighbours' LAST pass (needed before rtdd_strip_finish / prolongation read the ghost rows). */
int rtdd_ipc_export(rtdd_ctx *ctx, void *handle64);
int rtdd_ipc_import(rtdd_ctx *ctx, const void *handle64, void **peerArena);
int rtdd_arena(rtdd_ctx *ctx, void **base, size_t *bytes);
int rtdd_strip_set_peers(rtdd_ctx *ctx, void *arenaAbove, void *arenaBelow);
int rtdd_strip_neighbours(rtdd_ctx *ctx, int level, int ownBegin, int ownEnd, int halo, int aboveWinBegin, int belowWinBegin);
int rtdd_strip_wait(rtdd_ctx *ctx, int level);
/* Staged peer exchange (rtdd_set_tuning("strip_peer_staging", 1) before rtdd_strip_neighbours): the passes stay the plain
 * sweep kernels; rtdd_strip_push copies the `halo` rows next to each strip boundary into the neighbours' staging areas
 * (peer memory) and raises their sequence flags, rtdd_strip_pull waits for the neighbours' flags and unpacks the staged
 * rows into this rank's ghost rows.  Call push, then pull, once per exchange; every rank must do the same number of
 * exchanges per level.  No NCCL call, no host round trip. */
int rtdd_strip_push(rtdd_ctx *ctx, int level);
int rtdd_strip_pull(rtdd_ctx *ctx, int level);
/* on = 0: the following passes of `level` keep their boundary rows to themselves (the finest level's last pass: nobody
 * reads the ghost rows afterwards); the flags are still raised.  Reset to on by rtdd_strip_neighbours. */
int rtdd_strip_push_enable(rtdd_ctx *ctx, int level, int on);
/* The level's LAST pass writing straight into the caller's pitched depth plane and, if depthU8 is non-null, the 8-bit map
 * (GpuMat::convertTo, ref: src/main.cpp:290): rtdd_strip_pass + rtdd_strip_finish in one where no halo exchange follows (the
 * finest level).  depth / depthU8 are the FULL planes (row 0 = row 0 of the level, 16-byte aligned rows); every row of the
 * window is written, ghost rows with their stale values. */
int rtdd_strip_pass_to(rtdd_ctx *ctx, int level, int firstSweep, int nsweeps, int haloT, float *depth, size_t depthPitch,
                       uint8_t *depthU8, size_t depthU8Pitch);
/* cv::pyrUp restricted to destination rows [rowBegin, rowEnd); src and dst are the full planes */
int rtdd_pyrup_depth_rows(rtdd_ctx *ctx, const float *src, size_t srcPitch, int srcRows, int srcCols,
                          float *dst, size_t dstPitch, int dstRows, int dstCols, int rowBegin, int rowEnd);

/* ---- GPUImageProcessing -------------------------------------------------- */

/* replaces GPUConvertToFloat     ref: include/GPUImageProcessing.h:4-5, src/GPUImageProcessing.cu:8-21,72-79 */
int rtdd_convert_to_float(rtdd_ctx *ctx, const uint8_t *src, size_t srcPitch, float *dst, size_t dstPitch,
                          const uint8_t *mask, size_t maskPitch, int rows, int cols);
/* replaces GPUPyrDownAnnotation  ref: include/GPUImageProcessing.h:6-8, src/GPUImageProcessing.cu:23-49,81-91 */
int rtdd_pyrdown_annotation(rtdd_ctx *ctx, const uint8_t *prevScribble, size_t prevScribblePitch,
                            const uint8_t *prevEdited, size_t prevEditedPitch, int previousRows, int previousCols,
                            uint8_t *currScribble, size_t currScribblePitch,
                            uint8_t *currEdited, size_t currEditedPitch, int currentRows, int currentCols);
/* replaces GPUPaintImage         ref: include/GPUImageProcessing.h:9-10, src/GPUImageProcessing.cu:51-70,93-100 */
int rtdd_paint(rtdd_ctx *ctx, int x, int y, int scribbleColor, int scribbleRadius,
               uint8_t *edited, size_t editedPitch, uint8_t *scribble, size_t scribblePitch, int rows, int cols);

/* replaces the host loop that turns a loaded annotation into the two planes the solver works on
 * ref: src/main.cpp:160-170 (and :158 edited = the image, :132 scribble = 0).  `annotation` is ONE u8 plane, 32 = not annotated:
 * every pixel != 32 gets edited B = G = R = that value and scribble = 255, every other pixel edited = bgr and scribble = 0.
 * All four planes are device planes and must not overlap. */
int rtdd_annotation_ingest(rtdd_ctx *ctx, const uint8_t *annotation, size_t annotationPitch, const uint8_t *bgr, size_t bgrPitch,
                           uint8_t *edited, size_t editedPitch, uint8_t *scribble, size_t scribblePitch, int rows, int cols);

/* ---- GPUDepthEffect ------------------------------------------------------ */

/* replaces GPUSimulateDesaturation  ref: include/GPUDepthEffect.h:6-7, src/GPUDepthEffect.cu:8-27,95-103 */
int rtdd_desaturate(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                    const float *depth, size_t depthPitch, uint8_t *out, size_t outPitch, int rows, int cols);
/* replaces GPUSimulateHaze          ref: include/GPUDepthEffect.h:8-9, src/GPUDepthEffect.cu:74-93,115-123 */
int rtdd_haze(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
              uint8_t *out, size_t outPitch, int rows, int cols);
/* replaces GPUSimulateDefocus       ref: include/GPUDepthEffect.h:4-5, src/GPUDepthEffect.cu:29-72,105-113 */
int rtdd_defocus(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                 uint8_t *out, size_t outPitch, int rows, int cols);
/* All three effects from one read of image + gray + depth (north_star subsystem 3). */
int rtdd_effects_fused(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                       const float *depth, size_t depthPitch,
                       uint8_t *desat, size_t desatPitch, uint8_t *haze, size_t hazePitch,
                       uint8_t *defocus, size_t defocusPitch, int rows, int cols);

/* DepthEffect on rows [rowBegin, rowEnd) only (row strips across GPUs, SURVEY.md section 8e row 3): every plane is the FULL image
 * plane, any of the three outputs may be NULL, and only the strip's rows of the outputs are written -- with exactly the bytes
 * the whole-image calls put there (defocus: K from the full image's diagonal, ref: src/GPUDepthEffect.cu:42; its summed-area
 * table is built over the strip plus half a box on each open side). */
int rtdd_effects_rows(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                      const float *depth, size_t depthPitch, uint8_t *desat, size_t desatPitch, uint8_t *haze, size_t hazePitch,
                      uint8_t *defocus, size_t defocusPitch, int rows, int cols, int rowBegin, int rowEnd);

/* Extension, no reference counterpart: depth-of-field refocus of a device image by a device depth plane (see DESIGN.md §7).
 * Per pixel, with d' = depth clamped to [0, 255] (NaN -> 0): e = max(|d' - focusDepth| - depthOfField, 0),
 * a = (int)((double)((float)aperture * e) / 255.0), h = a / 2; h = 0 copies the pixel, otherwise every channel is the floor of
 * the exact mean of orig over [y-h, y+h) x [x-h, x+h) clipped to the image.  focusDepth in [0, 255]; depthOfField (the half-width
 * of the sharp band, depth units) finite and >= 0; aperture (the largest box side, pixels) <= 4096, a negative one selects the
 * reference defocus's K = (int)(0.025 x diagonal).  focusDepth = 0, depthOfField = 0, aperture = K gives rtdd_defocus's bytes
 * for every depth <= 255 while K <= 257.  Builds the summed-area table of orig (4 launches, 5 for cols > 16384) and refocuses (1). */
int rtdd_refocus(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                 uint8_t *out, size_t outPitch, int rows, int cols, float focusDepth, float depthOfField, int aperture);

/* Extension, no reference counterpart: stereo views of a device image by a device depth plane, the image taken as the centre view
 * (see DESIGN.md §7).  Depth 0 is near, 255 far.  convergenceDepth c in [0, 255] is the zero-parallax plane; maxDisparity D, in
 * [0, RTDD_STEREO_MAX_DISPARITY] pixels, is the parallax of a depth 255 away from it.  Per source pixel (x, y):
 *   d' = fminf(fmaxf(d, 0), 255) (NaN -> 0; -0 counts as +0);
 *   s = cvt.rzi.s32.f64((double)__fmul_rn((float)D, __fsub_rn(d', c)) / 255.0), the signed parallax in [-D, D];
 *   hL = s / 2 (C division, toward zero), hR = s - hL; the pixel lands on tL = x - hL in the left view and on tR = x + hR in the
 *   right one (tR - tL = s: farther than c is behind the screen, nearer is in front).  Targets outside [0, cols) are dropped.
 * Per view, row and target column t:
 *   covered (a source lands on t): the source with the smallest d' wins (the nearest occludes) and t shows orig[y][winner].
 *     Two sources with equal d' have equal s, so they never land on the same target: the winner is unique, every order of
 *     evaluation gives the same bytes, and an atomic minimum over d' is exact;
 *   a hole, with l and r the nearest covered targets left and right of t in the row: t shows the view's pixel at l when l exists
 *     and (r does not, or d' of l's winner >= d' of r's winner), otherwise the view's pixel at r -- the farther side, the
 *     background, fills the hole, ties to the left;
 *   a row with no covered target (D large against cols): orig[y][t].
 * The anaglyph (red-cyan) takes B and G from the right view and R from the left one.  D = 0, or every depth equal to c, gives
 * left = right = anaglyph = orig; a constant depth d0 != c shifts the image by -hL / +hR and repeats the nearest covered column.
 * Outputs are device BGR planes with byte pitches >= 3 x cols; any of them may be NULL, not all three.  Side by side is pointers
 * alone: left = buf, right = buf + 3 x cols, both with pitch 6 x cols.  Outputs must not overlap orig or depth.  depth is an fp32
 * plane: its address and pitch are multiples of 4.  cols <= RTDD_STEREO_MAX_COLS (one row is held on chip).  One launch, no
 * context scratch. */
#define RTDD_STEREO_MAX_DISPARITY 1024
#define RTDD_STEREO_MAX_COLS      16384
int rtdd_stereo(rtdd_ctx *ctx, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                uint8_t *left, size_t leftPitch, uint8_t *right, size_t rightPitch, uint8_t *anaglyph, size_t anaglyphPitch,
                int rows, int cols, float convergenceDepth, int maxDisparity);

/* ---- pyramid ops either side of the path (SURVEY.md section 8f) ------------------- */

/* cv::cvtColor(BGR2GRAY)                 ref: src/main.cpp:111,138 */
int rtdd_bgr2gray(rtdd_ctx *ctx, const uint8_t *bgr, size_t bgrPitch, uint8_t *gray, size_t grayPitch, int rows, int cols);
/* cv::pyrDown on the u8 gray plane       ref: src/main.cpp:112,143-145,244-246; dst is ceil(rows/2) x ceil(cols/2) */
int rtdd_pyrdown_gray(rtdd_ctx *ctx, const uint8_t *src, size_t srcPitch, int srcRows, int srcCols,
                      uint8_t *dst, size_t dstPitch);
/* cv::pyrUp on the fp32 depth plane      ref: src/main.cpp:272-279; dst is 2n or 2n+1 in each dimension */
int rtdd_pyrup_depth(rtdd_ctx *ctx, const float *src, size_t srcPitch, int srcRows, int srcCols,
                     float *dst, size_t dstPitch, int dstRows, int dstCols);
/* GpuMat::convertTo(CV_8UC1)             ref: src/main.cpp:290 (round half to even, saturate) */
int rtdd_quantise_u8(rtdd_ctx *ctx, const float *src, size_t srcPitch, uint8_t *dst, size_t dstPitch, int rows, int cols);

/* ---- one whole frame, the body of main.cpp's 'd'/--live branch ------------ */

/* ref: src/main.cpp:232-295.  The context owns device copies of the per-level gray,
 * scribble, edited and depth planes (what main.cpp keeps in its GpuMat vectors).
 * rtdd_frame_set_image uploads the level-0 BGR image from HOST memory and builds
 * the gray pyramid (main.cpp:111-112,138-147); it also resets the depth planes to
 * 255 and the annotation planes to 0 (main.cpp:130-136). */
int rtdd_frame_set_image(rtdd_ctx *ctx, const uint8_t *bgrHost, size_t bgrPitch);
/* One frame: upload level-0 scribble mask + edited image from HOST (main.cpp:236-237),
 * restrict annotations (:249), inject (:257,281), solve every level coarse to fine
 * (:261-288) with maxIterations at the coarsest level, quantise (:290) and download the
 * u8 depth map to HOST (:291).  depthU8Host may be NULL (no download).  A depthU8Host in pinned (page-locked) memory with a
 * 4-byte aligned base and pitch is written by the last sweep pass itself, over PCIe while it computes; any other plane is
 * filled by a copy after the last pass.  Either way the map is complete when the call returns. */
int rtdd_frame_solve_host(rtdd_ctx *ctx, const uint8_t *scribbleHost, size_t scribblePitch,
                          const uint8_t *editedHost, size_t editedPitch,
                          int maxIterations, uint8_t *depthU8Host, size_t depthU8Pitch);
/* The same frame from the reference's persistent annotation format (the -a file, ref: src/main.cpp:160-170): ONE u8 HOST plane,
 * 32 = not annotated.  Uploads 1 B/px instead of 4 B/px and expands it on the device (rtdd_annotation_ingest) into the
 * context's level-0 scribble / edited planes; otherwise identical to rtdd_frame_solve_host. */
int rtdd_frame_solve_host_annotation(rtdd_ctx *ctx, const uint8_t *annotationHost, size_t annotationPitch, int maxIterations,
                                     uint8_t *depthU8Host, size_t depthU8Pitch);
/* ref: src/main.cpp:291 -- download of the 8-bit depth map of the last solved frame into HOST memory.  sync = 0 leaves the copy
 * in flight on the context stream (batch mode: one host thread keeps several contexts busy and synchronises them later). */
int rtdd_frame_read_depth_u8(rtdd_ctx *ctx, uint8_t *depthU8Host, size_t depthU8Pitch, int sync);
/* Same frame with the annotation planes already on the device (paint with
 * rtdd_frame_paint); nothing crosses PCIe. */
int rtdd_frame_solve(rtdd_ctx *ctx, int maxIterations);
/* The live loop's frame (ref: src/main.cpp:232-295 with the strokes painted on the device by rtdd_frame_paint): rtdd_frame_solve
 * followed by the download of the 8-bit map (main.cpp:291) into HOST memory -- stored by the last level-0 pass itself when
 * depthU8Host is pinned and 4-byte aligned ("zero_copy_out"), a copy after the last pass otherwise.  Returns after the map is
 * complete. */
int rtdd_frame_solve_download(rtdd_ctx *ctx, int maxIterations, uint8_t *depthU8Host, size_t depthU8Pitch);
/* Warm-start incremental re-solve for live strokes (extension; the reference's only warm start is the coarsest depth
 * plane persisting between frames, ref: src/main.cpp:257).  Levels coarser than `coarsestLevel` are skipped; level
 * `coarsestLevel` starts from ITS OWN previous solution with the current annotations re-imposed and runs its scheduled
 * sweeps; finer levels proceed as in rtdd_frame_solve.  coarsestLevel = levels-1 is exactly rtdd_frame_solve. */
int rtdd_frame_solve_incremental(rtdd_ctx *ctx, int maxIterations, int coarsestLevel);
/* Extension, NOT parity (the reference always re-solves the whole pyramid, ref: src/main.cpp:232-295): a frame after an edit that
 * touched level-0 rows [rowBegin, rowEnd) only (a brush stroke).  Coarse levels -- every level below 2^20 pixels, and every level
 * the band of rows (scaled to the level, widened by `dilation` rows per side) covers by >= 60 % -- are solved whole and equal
 * the parity frame; on the large levels only the band is re-solved between two frozen rows of the previous solution, and the
 * rows outside receive the prolongated change of the coarser level.  How far the result is from the parity frame depends on the image
 * and the edit: tools/live_strokes.py reports it (8-bit identical fraction, mean |delta|).  Needs a previous frame. */
int rtdd_frame_solve_band(rtdd_ctx *ctx, int maxIterations, int rowBegin, int rowEnd, int dilation);
/* ref: src/main.cpp:190-230 -- desaturation / haze / defocus of the frame image by the frame's solved depth, written to
 * caller-owned DEVICE planes (BGR u8, byte pitches; any of the three may be NULL).  The defocus summed-area table depends
 * on the image only and is built once per rtdd_frame_set_image, not once per call. */
int rtdd_frame_effects(rtdd_ctx *ctx, uint8_t *desat, size_t desatPitch, uint8_t *haze, size_t hazePitch, uint8_t *defocus, size_t defocusPitch);
/* rtdd_refocus on the frame context's own image and solved level-0 depth, with the cached summed-area table (shared with
 * rtdd_frame_effects): 1 launch, plus the table's 4 (5 for cols > 16384) when it is absent.
 * focusX, focusY inside the image: focus = clamped depth under that pixel, read on the device (focusDepth ignored) -- a graph
 * captured from this call follows every later solve;  focusX = focusY = -1: focus = focusDepth. */
int rtdd_frame_refocus(rtdd_ctx *ctx, uint8_t *out, size_t outPitch, int focusX, int focusY, float focusDepth,
                       float depthOfField, int aperture);
/* rtdd_stereo on the frame context's own image and solved level-0 depth (1 launch; the summed-area table cached for
 * rtdd_frame_effects / rtdd_frame_refocus is left valid).
 * convergenceX, convergenceY inside the image: c = clamped depth under that pixel, read on the device (convergenceDepth ignored)
 * -- a graph captured from this call follows every later solve;  convergenceX = convergenceY = -1: c = convergenceDepth. */
int rtdd_frame_stereo(rtdd_ctx *ctx, uint8_t *left, size_t leftPitch, uint8_t *right, size_t rightPitch,
                      uint8_t *anaglyph, size_t anaglyphPitch, int convergenceX, int convergenceY,
                      float convergenceDepth, int maxDisparity);
/* ref: src/main.cpp:46-62 -- brush stroke into the context's level-0 annotation planes */
int rtdd_frame_paint(rtdd_ctx *ctx, int x, int y, int scribbleColor, int scribbleRadius);
/* device pointers/pitches of the context-owned planes (for effects, tests, downloads) */
int rtdd_frame_plane(rtdd_ctx *ctx, int which, int level, void **ptr, size_t *pitch, int *rows, int *cols);
#define RTDD_PLANE_DEPTH    0   /* fp32 */
#define RTDD_PLANE_GRAY     1   /* u8, ceil-sized like cv::pyrDown's output */
#define RTDD_PLANE_SCRIBBLE 2   /* u8 mask, 255 = annotated */
#define RTDD_PLANE_EDITED   3   /* u8 x 3 */
#define RTDD_PLANE_BGR      4   /* u8 x 3, level 0 only */
#define RTDD_PLANE_DEPTH_U8 5   /* u8, level 0 only */

/* rtdd_frame_set_image for a BGR image that already lives on the device (pitched, rows x 3*cols bytes). */
int rtdd_frame_set_image_device(rtdd_ctx *ctx, const uint8_t *bgrDevice, size_t bgrPitch);

/* ---- one frame of ONE image across several GPUs, row strips (BASELINE configs[4]); no reference counterpart ---------------
 * The frame loop is main.cpp's (ref: src/main.cpp:232-295).  Every rank = one context on one GPU holding the whole image and
 * annotation planes (rtdd_frame_set_image*, rtdd_frame_plane); levels of at least minStripPixels pixels are cut into row
 * strips (rtdd_plan_strips), the coarser ones are solved by every rank.  Halo rows (`halo` per open side, passes of
 * `passSweeps` sweeps between two exchanges) travel through peer memory (rtdd_strip_set_peers with the neighbours' arenas:
 * rtdd_arena inside one process after cudaDeviceEnablePeerAccess, rtdd_ipc_export / _import between processes).  All ranks
 * must issue the same calls.  Owned rows are bit-identical to the one-GPU frame. */
int rtdd_strip_frame_setup(rtdd_ctx *ctx, int rank, int nranks, int halo, int passSweeps, long long minStripPixels);
int rtdd_strip_frame_solve(rtdd_ctx *ctx, int maxIterations);
/* SURVEY.md 8d config 5 (i): only the finest level, `sweeps` sweeps from the guess its depth plane holds */
int rtdd_strip_frame_level0(rtdd_ctx *ctx, int sweeps);
/* this rank's rows of `level`: *split = 0 if the level is solved whole by every rank; own rows [ownBegin, ownEnd), window incl. ghosts */
int rtdd_strip_frame_rows(rtdd_ctx *ctx, int level, int *split, int *ownBegin, int *ownEnd, int *winBegin, int *winEnd);
/* ref: src/main.cpp:190-230 on this rank's rows of the finest level; outputs are FULL device planes, only owned rows are written */
int rtdd_strip_frame_effects(rtdd_ctx *ctx, uint8_t *desat, size_t desatPitch, uint8_t *haze, size_t hazePitch, uint8_t *defocus, size_t defocusPitch);

/* ---- several GPUs from ONE process: one host thread per GPU inside the library (what a C++ host like main.cpp links) -------
 * rtdd_mgpu_create makes one context per listed device, enables peer access between neighbours and wires their arenas.
 * halo / passSweeps / minStripPixels <= 0 select the defaults (16 / 8 / 2^22).  Every call below runs on all GPUs concurrently
 * and returns when all have finished; *msDevice (may be NULL) = the slowest rank's device time.  A handle serves ONE calling
 * thread at a time (the command slot is shared by the worker threads); different handles are independent. */
typedef struct rtdd_mgpu rtdd_mgpu;
int rtdd_mgpu_create(const int *devices, int ndevices, int rows, int cols, int levels, float beta, int halo, int passSweeps,
                     long long minStripPixels, rtdd_mgpu **out);
int rtdd_mgpu_destroy(rtdd_mgpu *m);
int rtdd_mgpu_devices(const rtdd_mgpu *m);
const char *rtdd_mgpu_last_error(const rtdd_mgpu *m);
rtdd_ctx *rtdd_mgpu_context(rtdd_mgpu *m, int rank);
/* configs[4]: the image (HOST, BGR) goes to every GPU; a frame = annotation plane in (HOST, 32 = not annotated), 8-bit map out */
int rtdd_mgpu_set_image(rtdd_mgpu *m, const uint8_t *bgrHost, size_t bgrPitch);
int rtdd_mgpu_frame_solve_host_annotation(rtdd_mgpu *m, const uint8_t *annotationHost, size_t annotationPitch, int maxIterations,
                                          uint8_t *depthU8Host, size_t depthU8Pitch, float *msDevice);
int rtdd_mgpu_frame_solve(rtdd_mgpu *m, int maxIterations, float *msDevice);      /* annotations already on the devices */
int rtdd_mgpu_level0(rtdd_mgpu *m, int sweeps, float *msDevice);
/* configs[3]: nimages independent images, image i on GPU i mod N, every image a full job from HOST buffers */
int rtdd_mgpu_batch_solve(rtdd_mgpu *m, int nimages, const uint8_t *const *bgrHost, size_t bgrPitch, const uint8_t *const *annotationHost,
                          size_t annotationPitch, int maxIterations, uint8_t *const *depthU8Host, size_t depthU8Pitch, float *msDevice);

#ifdef __cplusplus
}
#endif
#endif /* RTDD_H */
