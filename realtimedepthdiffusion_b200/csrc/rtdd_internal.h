// Internal declarations shared by the translation units of librtdd.so.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include <map>
#include <tuple>
#include <string>
#include <vector>

#include "rtdd.h"

// One pyramid level's scratch in the HBM arena.  Float planes share one row pitch
// (pitchF floats, a multiple of 64 => rows start 256 B aligned, TMA-legal); byte
// planes share pitchB (a multiple of 128).  Padding columns/rows are zero.
struct RtddLevel {
    int rows = 0, cols = 0;
    int planeRows = 0;         // rows the level's planes can hold: `rows`, or -- contexts made by rtdd_create_strip -- the largest row
                               // window any rank keeps of a split level (the same on every rank, so the arenas have one layout)
    int pitchF = 0;            // floats per row of x[] planes
    int pitchB = 0;            // bytes per row of link/mask planes
    float *x[4] = {nullptr, nullptr, nullptr, nullptr};   // rotating iterate planes
    uint8_t *linkR = nullptr;  // LUT index of link (x,y)-(x+1,y)
    uint8_t *linkD = nullptr;  // LUT index of link (x,y)-(x,y+1)
    uint8_t *mask = nullptr;   // 0xFF where the scribble plane == 255 (Dirichlet), else 0
    // TMA descriptors of the planes above (128x64-element boxes), built once in rtdd_create
    CUtensorMap tmX[4], tmLinkR, tmLinkD, tmMask;
    CUtensorMap tmLinkD1;      // linkD as 144 x 65 boxes: the cluster form loads the row above its tile as well
    bool hasMaps = false;
    // events bracketing the most recent sweep graph of this level (rtdd_level_sweep_ms)
    cudaEvent_t evBegin = nullptr, evEnd = nullptr;
    bool timed = false;
    int lastIters = 0, lastKernels = 0;
    // row-strip mode (rtdd_strip_*): the level's planes hold rows [stripBegin, stripBegin + stripRows) of the level
    int stripBegin = 0, stripRows = 0, stripPair = 0;
    // fused halo push (rtdd_strip_neighbours): geometry of this rank's strip and of its neighbours' windows
    bool stripFused = false, stripPushOff = false;
    int stripOwnBegin = 0, stripOwnEnd = 0, stripHalo = 0, stripUpWinBegin = -1, stripDnWinBegin = -1;
    unsigned int stripPassAbs = 0, stripFirstPassAbs = 0, stripCtaAbs = 0;   // monotonically increasing tickets
    unsigned int *dStripWords = nullptr;   // [0] CTA ticket, [1] flag written by the rank above, [2] flag written by the rank below;
                                           // staged exchange: [4] push-kernel ticket, [5] sequence pushed by the rank above, [6] ... below
    // staged peer exchange (rtdd_strip_push / rtdd_strip_pull): [buffer 2][from above, from below][x_k, x_{k-1}][RTDD_MAX_HALO rows]
    float *stage = nullptr;
    unsigned int peerSeq = 0;              // exchanges done so far on this level (monotonic; identical on every rank)
    unsigned int *dResidual = nullptr;   // bits of the max-norm of the last sweep's update (rtdd_level_residual)
    unsigned int *dBad = nullptr;        // != 0: the level's start iterate holds a value beyond +-4096 or a NaN (set by the level set-up kernel,
                                         // cleared by a memset before it): the sweeps then divide the IEEE way
    unsigned int *dPeerBad = nullptr;    // row strips with the staged exchange: the same verdict of the neighbouring ranks (sticky; set by their
                                         // push kernels over NVLink); null otherwise
    bool magnitudeCheck = false;         // row-strip windows WITHOUT that exchange of verdicts (NCCL / fused modes): every pass scans its own tiles
    bool stripScan = false;              // (state of the level's current strip: see rtdd_strip_init / rtdd_strip_neighbours)
};

// Context-owned images of the frame driver (what main.cpp keeps in GpuMat vectors).
struct RtddFrameLevel {
    int rows = 0, cols = 0;        // floor sizes (depth / scribble / edited)
    int grayRows = 0, grayCols = 0; // ceil sizes (cv::pyrDown output)
    float *depth = nullptr;   size_t depthPitch = 0;
    uint8_t *gray = nullptr;  size_t grayPitch = 0;
    uint8_t *scribble = nullptr; size_t scribblePitch = 0;
    uint8_t *edited = nullptr;   size_t editedPitch = 0;
};

struct RtddGraphKey {
    int kind;            // 1 = one level (rtdd_solve_level), 2 = whole frame (rtdd_frame_solve)
    int level, iters, variant, T;
    const void *p[3];    // caller planes baked into the graph: depth, scribble, gray
    size_t pitch[3];
    bool operator<(const RtddGraphKey &o) const
    {
        return std::tie(kind, level, iters, variant, T, p[0], p[1], p[2], pitch[0], pitch[1], pitch[2]) <
               std::tie(o.kind, o.level, o.iters, o.variant, o.T, o.p[0], o.p[1], o.p[2], o.pitch[0], o.pitch[1], o.pitch[2]);
    }
};

struct RtddLevelTiming { int level, iters, kernels; };
struct RtddGraph {
    cudaGraphExec_t exec = nullptr;
    int kernels = 0;
    int resultPlane = 0;   // index into RtddLevel::x holding x_K after the graph ran
    std::vector<RtddLevelTiming> timing;   // what rtdd_level_sweep_ms reports after THIS graph ran (copied into the levels at every launch)
};

// one rank's share of a row-strip frame (rtdd_strip_frame_*): the decomposition of every level, as planned by rtdd_plan_strips
struct RtddStripFrame {
    bool ready = false;
    int rank = 0, nranks = 1, halo = 16, passSweeps = 8;
    std::vector<int> split, ownBegin, ownEnd;      // per level; own ranges indexed [level * nranks + rank]
};

struct rtdd_ctx {
    int device = 0;
    int rows = 0, cols = 0, levels = 0;
    int smCount = 148;
    cudaStream_t ownStream = nullptr;
    cudaStream_t stream = nullptr;
    cudaStream_t captureStream = nullptr;   // private non-blocking stream used only to capture sweep graphs
    void *arena = nullptr;
    size_t arenaBytes = 0;
    std::vector<RtddLevel> lv;
    float *dLut = nullptr;       // 257 floats
    float hLut[257];
    bool lutLoaded = false;
    int variant = 0;             // 0 auto, 1 single-sweep, 2 temporally blocked, 3 cluster-resident
    char *peerUp = nullptr, *peerDn = nullptr;   // neighbours' arenas (IPC-mapped or same-process), same layout as `arena`
    std::vector<void *> ipcImports;              // arenas mapped by rtdd_ipc_import (closed in rtdd_destroy)
    unsigned int *dErrWord = nullptr;            // device word: RTDD_SPIN_TIMED_OUT once a halo wait gave up
    unsigned int *dPeerBadWord = nullptr;        // device word: a neighbouring rank saw an iterate beyond +-4096 (sticky, see RtddLevel::dPeerBad)
    unsigned int spinTimeoutMs = 20000;          // rtdd_set_tuning("spin_timeout_ms", ...)
    float *dOmega = nullptr;     // the omega schedule (prefix-stable), dOmegaCap entries
    int dOmegaCap = 0;
    int sweepsPerPass = 0;       // 0 auto
    std::vector<int> passPlan[32];   // per level: the caller's own pass lengths (rtdd_set_pass_plan; empty = the planner's)
    bool planThroughput = false;     // pass plans minimise total SM time instead of the level's latency (contexts of a batch; "plan_throughput")
    std::map<RtddGraphKey, RtddGraph> graphs;
    std::vector<RtddLevelTiming> captureTiming;   // filled by enqueue_level while a graph is being captured
    unsigned long long launches = 0;
    std::string err;
    // frame driver state
    std::vector<RtddFrameLevel> fl;
    void *frameArena = nullptr;
    uint8_t *bgr = nullptr; size_t bgrPitch = 0;
    uint8_t *depthU8 = nullptr; size_t depthU8Pitch = 0;
    uint8_t *annot = nullptr; size_t annotPitch = 0;      // level-0 single-plane annotation staging (rtdd_frame_solve_host_annotation)
    bool imageSet = false;
    bool stripResidual = false;        // rtdd_strip_pass also fills the level's residual word (+7 % per pass at 16K: only rtdd_solve_level_converge asks)
    bool peerStaging = false;          // rtdd_set_tuning("strip_peer_staging", 1): halo rows travel through rtdd_strip_push / _pull
    RtddStripFrame sf;
    bool frameSatValid = false;        // satScratch holds the summed-area table of the frame image (rtdd_frame_effects)
    // defocus scratch (summed-area tables), grown on demand
    void *satScratch = nullptr; size_t satBytes = 0;
    // rtdd_frame_solve_band: copies of the levels' previous solutions (levels 1 .. levels-1), same pitches as the frame's depth planes
    void *bandArena = nullptr;
    std::vector<float *> bandOld;
};

int rtdd_fail(rtdd_ctx *ctx, int code, const char *where);
int rtdd_check(rtdd_ctx *ctx, cudaError_t e, const char *where);

static inline int rtdd_div_up(int a, int b) { return (a + b - 1) / b; }
static inline size_t rtdd_round_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

// ---- kernel launchers (defined in the .cu translation units) ----------------
namespace rtdd {

// solver_kernels.cu
// A caller-visible destination for the LAST sweep pass of a level: the pitched depth plane (16-byte aligned rows)
// and optionally the 8-bit quantised map.  Null = the library's own planes.
struct SweepTarget {
    float *x; int pitchX;        // floats per row; null = keep the library's own planes
    uint8_t *u8; int pitchU8;    // may be null
    unsigned int *res;           // may be null: receives the bits of max |x_K - x_{K-1}| (atomicMax)
    uint8_t *u8b; int pitchU8b;  // may be null: a second copy of the 8-bit map (device alias of a pinned host plane); needs u8 != null
};
// fused multi-GPU halo push (solver_kernels.cu); plain data, filled by rtdd_strip_pass
struct HaloPush {
    float *upX, *upP, *dnX, *dnP;          // neighbour's (x_{k+1}, x_k) planes, window-local row 0; null = no such neighbour
    int upLo, upHi, upDelta;               // my window rows [upLo, upHi) land in neighbour row (row + upDelta)
    int dnLo, dnHi, dnDelta;
    int pitch;                             // floats per row (identical on every rank)
    int storeLo, storeHi;                  // only window rows [storeLo, storeHi) are stored locally: ghost rows that a neighbour
                                           // fills must not be overwritten with this rank's stale values
    unsigned int *counter;                 // this rank's CTA completion ticket (null = fused mode off)
    unsigned int doneTarget;               // ticket value once every CTA of this pass has finished
    unsigned int *upFlag, *dnFlag;         // flags in the neighbours' memory, set to flagValue by the last CTA
    unsigned int flagValue;
    const unsigned int *waitUp, *waitDn;   // this rank's flags: spin until >= waitValue before touching ghost rows (0 = no wait)
    unsigned int waitValue;
    unsigned int *err;                     // context error word: a wait that timed out stores RTDD_SPIN_TIMED_OUT here
    unsigned int timeoutMs;                // 0 = wait for ever
};
#define RTDD_SPIN_TIMED_OUT 0x51A1u
cudaError_t launch_level_prolong_init(cudaStream_t s, const RtddLevel &L, const float *src, size_t srcPitch, int srows, int scols,
                                      const uint8_t *edited, size_t editedPitch, const uint8_t *scribble, size_t scribblePitch,
                                      const uint8_t *gray, size_t grayPitch, int threshold, float *x0, unsigned int *residual);
cudaError_t launch_level_init(cudaStream_t s, const RtddLevel &L, const float *depth, size_t depthPitch,
                              const uint8_t *scribble, size_t scribblePitch,
                              const uint8_t *gray, size_t grayPitch, bool coarsest, int threshold, float *x0, unsigned int *residual = nullptr,
                              int fixRowA = -1, int fixRowB = -1);
cudaError_t launch_sweep_single(cudaStream_t s, const RtddLevel &L, const float *lut, const float *x, const float *prev,
                                float *out, float omega, float gamma, bool firstSweep, const SweepTarget *target = nullptr);
// temporally blocked: T sweeps (x, prev) -> (xOut, prevOut); omegas passed by value (<= RTDD_MAX_T)
#define RTDD_MAX_T 16
#define RTDD_MAX_HALO 32      // ghost rows per open strip side the staged peer exchange can carry
struct OmegaPack { float w[RTDD_MAX_T]; };
cudaError_t launch_sweep_blocked(cudaStream_t s, const RtddLevel &L, const float *lut, const float *x, const float *prev,
                                 float *xOut, float *prevOut, OmegaPack om, int T, int nsweeps, float gamma, bool firstSweep, int smCount,
                                 const SweepTarget *target = nullptr, struct HaloPush *push = nullptr, int form = 0);
void blocked_plan(int rows, int cols, int iters, int smCount, int *T, int *form);
int blocked_plan_passes(int rows, int cols, int iters, int smCount, int hostMap, int throughput, int *passes, int capacity, int *form);
// staged peer exchange: rows of (x_k, x_{k-1}) between this rank's planes and a staging area, plus the completion flags
struct HaloRows {
    const float *srcX, *srcP;     // first row to copy of each plane (null: nothing on this side)
    float *dstX, *dstP;
    int rows;
};
cudaError_t launch_halo_push(cudaStream_t s, HaloRows up, HaloRows dn, int pitchF, unsigned int *ticket,
                             unsigned int *upFlag, unsigned int *dnFlag, unsigned int flagValue,
                             const unsigned int *ownBad, const unsigned int *peerBadIn, unsigned int *upPeerBad, unsigned int *dnPeerBad);
cudaError_t launch_halo_pull(cudaStream_t s, HaloRows up, HaloRows dn, int pitchF, const unsigned int *waitUp, const unsigned int *waitDn,
                             unsigned int value, unsigned int *err, unsigned int timeoutMs);
cudaError_t launch_halo_wait(cudaStream_t s, const unsigned int *waitUp, const unsigned int *waitDn, unsigned int value,
                             unsigned int *err, unsigned int timeoutMs);
// per-device function attributes (cluster size, dynamic shared memory) of every kernel that needs them; called once per
// context from rtdd_create with the context's device current (no lazily initialised statics: contexts may be created
// from several host threads, one per GPU)
cudaError_t configure_kernels();
int blocked_max_T();
void set_blocked_tile_override(int tile);
void set_blocked_tma(int mode);
void set_blocked_cluster(int c);
void set_blocked_grid_cap(int cap);
void set_resident_warps(int w);
void set_resident_r1_max_warps(int w);
void set_pdl(int on);
int pdl_enabled();

// Programmatic dependent launch (sm_90+): the kernel may be scheduled while its predecessor in the stream drains; it orders
// itself against the predecessor's memory with griddepcontrol.wait (every kernel launched through here executes it before
// its first dependent access).  Captured into CUDA graphs as programmatic edges.
template <class Kernel, class... Args>
static inline cudaError_t launch_pdl(Kernel kernel, dim3 grid, dim3 block, size_t smemBytes, cudaStream_t s, Args... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smemBytes;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, args...);
}
// resident (one cluster, all sweeps in one launch); omegas = device array of nsweeps floats
bool resident_plan(int rows, int cols, int *R, int *clusterSize, int *blocksPerCta, int *WX);
cudaError_t launch_sweep_resident(cudaStream_t s, const RtddLevel &L, const float *lut, const float *x, float *xOut,
                                  const float *omegas, int nsweeps, float gamma, const SweepTarget *target = nullptr);
cudaError_t launch_division_selftest(cudaStream_t s, unsigned long long n, unsigned long long seed, int mode, unsigned long long *dMismatches);
cudaError_t launch_copy_out(cudaStream_t s, const RtddLevel &L, const float *x, float *depth, size_t depthPitch);
cudaError_t launch_export_links(cudaStream_t s, const RtddLevel &L, uint8_t *linkRight, uint8_t *linkDown, size_t outPitch);

// image_kernels.cu
cudaError_t launch_convert(cudaStream_t s, const uint8_t *src, size_t srcPitch, float *dst, size_t dstPitch,
                           const uint8_t *mask, size_t maskPitch, int rows, int cols);
cudaError_t launch_pyrdown_annotation(cudaStream_t s, const uint8_t *prevScribble, size_t prevScribblePitch,
                                      const uint8_t *prevEdited, size_t prevEditedPitch, int previousRows, int previousCols,
                                      uint8_t *currScribble, size_t currScribblePitch, uint8_t *currEdited, size_t currEditedPitch,
                                      int currentRows, int currentCols);
cudaError_t launch_annotation_ingest(cudaStream_t s, const uint8_t *ann, size_t annPitch, const uint8_t *bgr, size_t bgrPitch,
                                     uint8_t *edited, size_t editedPitch, uint8_t *scribble, size_t scribblePitch, int rows, int cols);
cudaError_t launch_paint(cudaStream_t s, int x, int y, int color, int radius, uint8_t *edited, size_t editedPitch,
                         uint8_t *scribble, size_t scribblePitch, int rows, int cols, int *launched);
cudaError_t launch_bgr2gray(cudaStream_t s, const uint8_t *bgr, size_t bgrPitch, uint8_t *gray, size_t grayPitch, int rows, int cols);
cudaError_t launch_pyrdown_gray(cudaStream_t s, const uint8_t *src, size_t srcPitch, int srows, int scols, uint8_t *dst, size_t dstPitch);
cudaError_t launch_pyrup_depth(cudaStream_t s, const float *src, size_t srcPitch, int srows, int scols,
                               float *dst, size_t dstPitch, int drows, int dcols);
cudaError_t launch_pyrup_depth_rows(cudaStream_t s, const float *src, size_t srcPitch, int srows, int scols,
                                    float *dst, size_t dstPitch, int drows, int dcols, int rowBegin, int rowEnd);
cudaError_t launch_band_prolong(cudaStream_t s, const float *newC, const float *oldC, size_t pitchC, int srows, int scols,
                                float *dst, size_t dstPitch, int drows, int dcols, int bandBegin, int bandEnd);
cudaError_t launch_quantise(cudaStream_t s, const float *src, size_t srcPitch, uint8_t *dst, size_t dstPitch, int rows, int cols);
cudaError_t launch_fill_f32(cudaStream_t s, float *dst, size_t pitch, int rows, int cols, float v);

// effect_kernels.cu
int defocus_kernel_size(int rows, int cols);
cudaError_t launch_desaturate(cudaStream_t s, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                              const float *depth, size_t depthPitch, uint8_t *out, size_t outPitch, int rows, int cols);
cudaError_t launch_haze(cudaStream_t s, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                        uint8_t *out, size_t outPitch, int rows, int cols);
int defocus_kernel_size(int rows, int cols);
size_t defocus_scratch_bytes(int rows, int cols);
// summed-area table of orig into `scratch`; *launched = number of kernels launched (4, or 5 wider than 16384 columns)
cudaError_t launch_sat_build(cudaStream_t s, void *scratch, const uint8_t *orig, size_t origPitch, int rows, int cols, int *launched);
// desat/haze may be null (defocus only); returns number of kernels launched through *launched
cudaError_t launch_defocus(cudaStream_t s, void *scratch, const uint8_t *orig, size_t origPitch, const uint8_t *gray, size_t grayPitch,
                           const float *depth, size_t depthPitch, uint8_t *defocus, size_t defocusPitch,
                           uint8_t *desat, size_t desatPitch, uint8_t *haze, size_t hazePitch,
                           int rows, int cols, int *launched, bool buildSat = true, int yBegin = 0, int yEnd = -1, int satRow0 = 0, int satRows = -1);
// depth-of-field refocus over a summed-area table that launch_sat_build left in `scratch` (one launch).  focusAt != null: the focus
// is the clamped depth at that device address, read by the kernel, and `focus` is ignored.  0 <= aperture <= RTDD_REFOCUS_MAX_APERTURE.
#define RTDD_REFOCUS_MAX_APERTURE 4096     // largest box side: windows stay <= 2^24 pixels, window sums < 2^32
cudaError_t launch_refocus(cudaStream_t s, const void *scratch, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                           uint8_t *out, size_t outPitch, int rows, int cols, float focus, const float *focusAt, float band, int aperture);
// stereo views and anaglyph (one launch, no scratch); any one or two of left / right / anaglyph may be null.  convAt != null: the
// convergence depth is the clamped depth at that device address, read by the kernel, and `conv` is ignored.
// 1 <= cols <= RTDD_STEREO_MAX_COLS, 0 <= maxDisparity <= RTDD_STEREO_MAX_DISPARITY.
cudaError_t launch_stereo(cudaStream_t s, const uint8_t *orig, size_t origPitch, const float *depth, size_t depthPitch,
                          uint8_t *left, size_t leftPitch, uint8_t *right, size_t rightPitch, uint8_t *anaglyph, size_t anaglyphPitch,
                          int rows, int cols, float conv, const float *convAt, int maxDisparity);
// the stereo kernel's shared-memory limit (a row of RTDD_STEREO_MAX_COLS columns); called next to configure_kernels
cudaError_t configure_stereo();

}  // namespace rtdd
