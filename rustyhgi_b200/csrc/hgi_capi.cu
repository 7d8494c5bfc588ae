// hgi_capi.cu -- the C ABI of libhgi_b200.so (include/hgi.h): context, pass planning, host/device
// entry points.  No CPU compute path exists here: every encode/decode/histogram goes through the
// CUDA kernels, and context creation fails when there is no sm_100 device.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <new>
#include <vector>

#include "../../include/hgi.h"
#include "hgi_device.cuh"
#include "hgi_kernels.h"

namespace {

constexpr int kSlots = 4;  // host-API pipeline: at most this many chunks in flight (H2D / kernels / D2H overlap)
// Slots actually used; HGI_B200_SLOTS overrides (tuning hook, 1..kSlots).
int slot_count()
{
    static const int v = [] {
        const char* e = std::getenv("HGI_B200_SLOTS");
        const long n = e ? std::atol(e) : 0;
        return (int)(n >= 1 && n <= kSlots ? n : 3);
    }();
    return v;
}
// Bytes per pipeline chunk of the host-pointer entry points; HGI_B200_CHUNK_MB overrides (tuning hook).
size_t chunk_bytes()
{
    static const size_t v = [] {
        const char* e = std::getenv("HGI_B200_CHUNK_MB");
        const long mb = e ? std::atol(e) : 0;
        return (size_t)(mb > 0 && mb <= 4096 ? mb : 64) << 20;
    }();
    return v;
}

// HGI_B200_POISON_SCRATCH=<0..255>: fill the device scratch planes with this byte before every launch chain (debug).
int poison_scratch()
{
    static const int v = [] {
        const char* e = std::getenv("HGI_B200_POISON_SCRATCH");
        return e && *e ? (int)(std::strtol(e, nullptr, 0) & 255) : -1;
    }();
    return v;
}

struct DevBuf {
    uint8_t* p = nullptr;
    size_t cap = 0;
};

// Device scratch of ONE stream's launch chain.  Chains on different streams may run at the same time (the slots of
// the host API, caller streams of the device API), so every stream owns its set: sharing one set let a chunk's fine
// pass read the next chunk's coarse planes.
struct Scratch {
    uint64_t gen = 0;    // bumped whenever one of the buffers moves: cached launch chains that point into them are stale
    DevBuf compact[4];   // ping-pong {recon, q} compact planes of the coarse passes
    DevBuf dec_in;       // decimated source of a coarse pass
    DevBuf region_in, region_out;   // scalable decode: the gathered window of the grid, and the decoded window
    // fork/join of the independent split launches of the quantizing encode (hgi_kernels.h PassArgs::side_stream)
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
};

struct Slot {
    cudaStream_t stream = nullptr;
    DevBuf in, out, aux, hist;
    Scratch scratch;
};

struct StreamScratch {
    cudaStream_t stream;
    Scratch scratch;
};

// A launch chain of the device API (decimate + coarse + fine [+ edge] [+ histogram] kernels of one call), captured
// once and replayed with one cudaGraphLaunch: what a caller with fixed buffers -- a frame loop, the band driver of
// the pool -- pays per call on the host drops from one launch per kernel to one launch per call.
struct ChainKey {
    int mode, interp, quant_kind, quant_level;
    const uint8_t* src;
    uint8_t *grid_out, *recon_out;
    uint32_t* hist;
    uint32_t n_images, w, h, pitch, levels;
    const Scratch* scratch;
    uint64_t scratch_gen;
    bool operator==(const ChainKey& o) const
    {
        return mode == o.mode && interp == o.interp && quant_kind == o.quant_kind &&
               quant_level == o.quant_level && src == o.src && grid_out == o.grid_out && recon_out == o.recon_out &&
               hist == o.hist && n_images == o.n_images && w == o.w && h == o.h && pitch == o.pitch &&
               levels == o.levels && scratch == o.scratch && scratch_gen == o.scratch_gen;
    }
};
struct ChainGraph {
    ChainKey key{};
    cudaGraphExec_t exec = nullptr;   // null: the chain was seen once and ran as plain launches
    uint64_t launches = 0;            // kernels in the chain
    uint64_t last_use = 0;
};
constexpr size_t kMaxChainGraphs = 16;
bool graphs_enabled()
{
    static const bool v = [] {
        const char* e = std::getenv("HGI_B200_GRAPHS");
        return !(e && e[0] == '0');
    }();
    return v;
}

constexpr size_t kMaxCallerStreams = 32;   // scratch sets kept for device-API caller streams; the oldest is recycled

}  // namespace

struct hgi_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaError_t last_err = cudaSuccess;
    uint64_t launches = 0;
    size_t chunk_bytes = 0;                       // host API pipeline (0: default / environment), see hgi_ctx_set_pipeline
    int n_slots = 0;
    std::vector<StreamScratch*> caller_scratch;   // device API: one scratch set per caller stream
    std::vector<ChainGraph> chains;               // device API: captured launch chains (see ChainKey)
    uint64_t chain_clock = 0, graph_launches = 0;
    Slot slots[kSlots];
    unsigned long long* d_metrics = nullptr;
};

// Several contexts (one per GPU of the box, in general) driven from one host thread: work is enqueued on every device
// before anything is waited for (SURVEY.md 8e: by image for batches, by row band for one huge plane).
struct hgi_pool {
    std::vector<hgi_ctx*> ctxs;
    std::vector<int> used;      // slot streams with work in flight, per context
};

namespace {

// Scope of one context's work: makes its device current (the caller's device is restored at the end) and charges the
// kernels launched inside the scope to it (hgi_ctx_kernel_launches).  Scopes nest: an inner scope takes its kernels
// out of hgi::launch_count(), so the outer one does not charge them again.
struct DeviceGuard {
    hgi_ctx* ctx;
    int prev = -1;
    bool ok = true;
    const uint64_t launched = hgi::launch_count();
    explicit DeviceGuard(hgi_ctx* c) : ctx(c)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != ctx->device) {
            cudaError_t e = cudaSetDevice(ctx->device);
            if (e != cudaSuccess) { ctx->last_err = e; ok = false; }
        }
    }
    ~DeviceGuard()
    {
        ctx->launches += hgi::launch_count() - launched;
        hgi::launch_count() = launched;
        if (prev >= 0) cudaSetDevice(prev);
    }
};

int fail(hgi_ctx* ctx, cudaError_t e)
{
    ctx->last_err = e;
    (void)cudaGetLastError();  // clear the sticky-free error state
    return e == cudaErrorMemoryAllocation ? HGI_ERR_ALLOC : HGI_ERR_CUDA;
}

#define HGI_CUDA(ctx, expr)                                  \
    do {                                                     \
        cudaError_t e__ = (expr);                            \
        if (e__ != cudaSuccess) return fail((ctx), e__);     \
    } while (0)

int reserve(hgi_ctx* ctx, DevBuf& b, size_t bytes)
{
    if (bytes <= b.cap) return HGI_OK;
    if (b.p) {
        HGI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (auto& s : ctx->slots)
            if (s.stream) HGI_CUDA(ctx, cudaStreamSynchronize(s.stream));
        HGI_CUDA(ctx, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    const size_t want = (bytes + 255) & ~(size_t)255;
    HGI_CUDA(ctx, cudaMalloc((void**)&b.p, want));
    b.cap = want;
    return HGI_OK;
}

void free_bufs(std::initializer_list<DevBuf*> bufs)
{
    for (DevBuf* b : bufs) {
        if (b->p) cudaFree(b->p);
        *b = DevBuf{};
    }
}

void destroy_side(Scratch& sc)
{
    if (sc.side) cudaStreamDestroy(sc.side);
    if (sc.ev_fork) cudaEventDestroy(sc.ev_fork);
    if (sc.ev_join) cudaEventDestroy(sc.ev_join);
    sc.side = nullptr;
    sc.ev_fork = sc.ev_join = nullptr;
}

void free_scratch(Scratch& sc)
{
    free_bufs({&sc.compact[0], &sc.compact[1], &sc.compact[2], &sc.compact[3], &sc.dec_in, &sc.region_in, &sc.region_out});
    destroy_side(sc);
}

// Stream of pipeline slot `k`, created on first use.
int slot_stream(hgi_ctx* ctx, int k)
{
    if (!ctx->slots[k].stream) HGI_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->slots[k].stream, cudaStreamNonBlocking));
    return HGI_OK;
}

// Waits for the streams of slots [0, n): nothing may still write into the caller's buffers when an entry point
// returns, on the error path too.  The first error (`rc`, else the first failed wait) is the one reported.
int drain(hgi_ctx* ctx, int n, int rc)
{
    for (int k = 0; k < n; ++k)
        if (ctx->slots[k].stream) {
            const cudaError_t e = cudaStreamSynchronize(ctx->slots[k].stream);
            if (e != cudaSuccess && rc == HGI_OK) rc = fail(ctx, e);
        }
    if (rc != HGI_OK) (void)cudaGetLastError();
    return rc;
}

// Scratch set of a device-API caller stream (created on first use).
Scratch* scratch_for(hgi_ctx* ctx, cudaStream_t st)
{
    for (size_t i = 0; i < ctx->caller_scratch.size(); ++i)
        if (ctx->caller_scratch[i]->stream == st) {
            if (i + 1 != ctx->caller_scratch.size()) {   // keep most-recently-used order
                StreamScratch* hit = ctx->caller_scratch[i];
                ctx->caller_scratch.erase(ctx->caller_scratch.begin() + (long)i);
                ctx->caller_scratch.push_back(hit);
            }
            return &ctx->caller_scratch.back()->scratch;
        }
    if (ctx->caller_scratch.size() >= kMaxCallerStreams) {
        // recycle the least recently used set: nothing of it may still be in flight (the stream may be gone: ignore errors)
        StreamScratch* old = ctx->caller_scratch.front();
        ctx->caller_scratch.erase(ctx->caller_scratch.begin());
        (void)cudaDeviceSynchronize();
        (void)cudaGetLastError();
        ++old->scratch.gen;              // chains captured for the old stream must not be replayed on the new one
        old->stream = st;
        ctx->caller_scratch.push_back(old);
        return &old->scratch;
    }
    StreamScratch* ss = new (std::nothrow) StreamScratch();
    if (!ss) return nullptr;
    ss->stream = st;
    ctx->caller_scratch.push_back(ss);
    return &ss->scratch;
}

int reserve(hgi_ctx* ctx, Scratch& sc, DevBuf& b, size_t bytes)
{
    if (bytes <= b.cap) return HGI_OK;
    ++sc.gen;
    return reserve(ctx, b, bytes);
}

// Prologue of a device-API call: the context's device for the call's duration, the caller's stream (NULL: the
// context's own) and, when asked for, that stream's scratch set.  A non-zero `rc` is the status to return.
struct DevCall {
    DeviceGuard g;
    cudaStream_t st;
    Scratch* sc = nullptr;
    int rc = HGI_OK;
    DevCall(hgi_ctx* ctx, void* stream, bool want_scratch = false)
        : g(ctx), st(stream ? (cudaStream_t)stream : ctx->stream)
    {
        if (!g.ok) rc = HGI_ERR_CUDA;
        else if (want_scratch && !(sc = scratch_for(ctx, st))) rc = HGI_ERR_ALLOC;
    }
};

int check_params(const hgi_params_t* p, bool encode)
{
    if (!p) return HGI_ERR_INVALID_ARG;
    if (p->levels > HGI_MAX_LEVELS) return HGI_ERR_INVALID_ARG;
    if (p->interp == HGI_INTERP_LINE || p->interp == HGI_INTERP_PREVIOUS) return HGI_ERR_UNSUPPORTED;
    if (p->interp != HGI_INTERP_CROSSED && p->interp != HGI_INTERP_LEFTTOP) return HGI_ERR_INVALID_ARG;
    if (encode) {
        if (p->quant_kind != HGI_QUANT_NOOP && p->quant_kind != HGI_QUANT_LINEAR) return HGI_ERR_INVALID_ARG;
        if (p->quant_kind == HGI_QUANT_LINEAR && (p->quant_level < 0 || p->quant_level > 3))
            return HGI_ERR_INVALID_ARG;
    }
    return HGI_OK;
}

// Levels whose sub-step is >= max(w,h) have no new points (only (0,0) lies on their lattice and
// it is a seed), so clamping `levels` leaves every byte unchanged (SURVEY.md Appendix A.1).
uint32_t effective_levels(uint32_t levels, uint32_t w, uint32_t h)
{
    const uint32_t m = w > h ? w : h;
    uint32_t need = 0;
    while (need < 32 && (1ull << need) < m) ++need;  // ceil(log2(m))
    return levels < need ? levels : need;
}

struct Pass {
    uint32_t d_log2, nlev;
};

// Split the hierarchy into passes of <= 4 levels, finest pass first in `out` order reversed later.
std::vector<Pass> plan_passes(uint32_t levels)
{
    std::vector<Pass> fine_to_coarse;
    uint32_t d = 0, rem = levels;
    while (rem > 0) {
        const uint32_t nl = rem < (uint32_t)hgi::kMaxPassLevels ? rem : (uint32_t)hgi::kMaxPassLevels;
        fine_to_coarse.push_back({d, nl});
        d += nl;
        rem -= nl;
    }
    return std::vector<Pass>(fine_to_coarse.rbegin(), fine_to_coarse.rend());
}

inline uint32_t ceil_shift(uint32_t v, uint32_t sh)
{
    return (uint32_t)(((uint64_t)v + (1ull << sh) - 1) >> sh);
}

inline bool aligned16(const void* p) { return ((uintptr_t)p & 15u) == 0; }

inline uint32_t align16(uint32_t v) { return (v + 15u) & ~15u; }

// mode: hgi::kModeEncode / kModeDecode.  All pointers are device pointers; planes have rows of `pitch` bytes.
int run_tile_path(hgi_ctx* ctx, Scratch& sc, int mode, const uint8_t* src, uint32_t n_images, uint32_t w, uint32_t h,
                  uint32_t pitch, uint32_t levels, const hgi_params_t* prm, uint8_t* grid_out, uint8_t* recon_out,
                  cudaStream_t st)
{
    const std::vector<Pass> passes = plan_passes(levels);
    const uint32_t qerr = (mode == hgi::kModeEncode) ? hgi::level_error(prm->quant_kind, prm->quant_level) : 0u;
    // compact planes (rows padded to 16 bytes): pass i (D>1) writes set (i&1), the next pass reads it
    size_t max_compact = 0;
    for (const Pass& ps : passes)
        if (ps.d_log2 > 0) {
            const size_t sz = (size_t)n_images * align16(ceil_shift(w, ps.d_log2)) * ceil_shift(h, ps.d_log2);
            if (sz > max_compact) max_compact = sz;
        }
    if (max_compact) {
        const int nbuf = passes.size() > 2 ? 4 : 2;
        for (int i = 0; i < nbuf; ++i) {
            if (mode == hgi::kModeDecode && (i & 1)) continue;  // decode carries no symbols
            int rc = reserve(ctx, sc, sc.compact[i], max_compact);
            if (rc) return rc;
        }
        int rc = reserve(ctx, sc, sc.dec_in, max_compact);
        if (rc) return rc;
    }
    // side stream + events for the split launches of the quantizing encode; created outside any capture (the first
    // sighting of a chain runs uncaptured), a single-image job gains most (the edge launches are one wave each)
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (mode == hgi::kModeEncode && qerr != 0 && !sc.side && st != cudaStreamLegacy &&
        cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusNone) {
        if (cudaStreamCreateWithFlags(&sc.side, cudaStreamNonBlocking) != cudaSuccess ||
            cudaEventCreateWithFlags(&sc.ev_fork, cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&sc.ev_join, cudaEventDisableTiming) != cudaSuccess) {
            (void)cudaGetLastError();
            destroy_side(sc);
        }
    }
    (void)cudaGetLastError();
    if (max_compact && poison_scratch() >= 0) {
        // debug hook (HGI_B200_POISON_SCRATCH=<byte>): the scratch planes start as a known pattern; results must not change
        for (auto& b : sc.compact)
            if (b.p) HGI_CUDA(ctx, cudaMemsetAsync(b.p, poison_scratch(), b.cap, st));
        HGI_CUDA(ctx, cudaMemsetAsync(sc.dec_in.p, poison_scratch(), sc.dec_in.cap, st));
    }
    const uint8_t* c_recon = nullptr;
    const uint8_t* c_q = nullptr;
    uint32_t ch = 0, cpitch = 0;
    for (size_t i = 0; i < passes.size(); ++i) {
        const Pass& ps = passes[i];
        hgi::PassArgs a{};
        a.src = src;
        a.w = w;
        a.h = h;
        a.pitch = pitch;
        a.d_log2 = ps.d_log2;
        a.nlev = ps.nlev;
        a.wD = ceil_shift(w, ps.d_log2);
        a.hD = ceil_shift(h, ps.d_log2);
        a.dpitch = align16(a.wD);
        a.ch = ch;
        a.cpitch = cpitch;
        a.c_recon = c_recon;
        a.c_q = c_q;
        a.n_images = n_images;
        a.quant_error = qerr;
        if (ps.d_log2 == 0) {
            a.grid_out = grid_out;
            a.recon_out = recon_out;
            if (st != cudaStreamLegacy && sc.side && sc.ev_fork && sc.ev_join) {
                a.side_stream = sc.side;
                a.ev_fork = sc.ev_fork;
                a.ev_join = sc.ev_join;
            }
            a.vec_ok = (pitch % 16 == 0) && aligned16(src) && (grid_out == nullptr || aligned16(grid_out)) &&
                       (recon_out == nullptr || aligned16(recon_out));
            if (a.vec_ok && (w % 16 != 0)) a.vec_ok = 2;   // padded rows: the last chunk of a row holds padding
        } else {
            const int set = (int)(i & 1) * 2;
            a.s_recon = sc.compact[set].p;
            a.s_q = sc.compact[set + 1].p;
            a.dec_in = sc.dec_in.p;
        }
        HGI_CUDA(ctx, hgi::launch_tile_pass(mode, prm->interp, a, st));
        c_recon = a.s_recon;
        c_q = a.s_q;
        ch = a.hD;
        cpitch = a.dpitch;
    }
    return HGI_OK;
}

int run_dev(hgi_ctx* ctx, Scratch& sc, int mode, const uint8_t* src, uint32_t n_images, uint32_t w, uint32_t h,
            uint32_t pitch, const hgi_params_t* prm, uint8_t* grid_out, uint8_t* recon_out, uint32_t* hist, cudaStream_t st)
{
    if (n_images == 0 || (size_t)w * h == 0) return HGI_OK;
    const uint32_t levels = effective_levels(prm->levels, w, h);
    uint8_t* primary = (mode == hgi::kModeEncode) ? grid_out : recon_out;
    if (levels == 0) {
        // L = 0: grid == image (src/encoder.rs:26-37 copies every pixel, the level loop is empty)
        HGI_CUDA(ctx, cudaMemcpy2DAsync(primary, pitch, src, pitch, w, (size_t)h * n_images, cudaMemcpyDeviceToDevice, st));
        if (mode == hgi::kModeEncode && recon_out)
            HGI_CUDA(ctx, cudaMemcpy2DAsync(recon_out, pitch, src, pitch, w, (size_t)h * n_images, cudaMemcpyDeviceToDevice, st));
    } else {
        int rc = run_tile_path(ctx, sc, mode, src, n_images, w, h, pitch, levels, prm, grid_out, recon_out, st);
        if (rc) return rc;
    }
    if (hist) {
        // The residual histogram is a pass of its own over the finished grid (hgi_hist_kernel, DESIGN.md 4.6)
        HGI_CUDA(ctx, hgi::launch_histogram(grid_out, w, h, pitch, n_images, hist, st));
    }
    return HGI_OK;
}

void drop_chain(ChainGraph& g)
{
    if (g.exec) cudaGraphExecDestroy(g.exec);
    g = ChainGraph{};
}

// run_dev for the device API: identical consecutive calls (same buffers, same parameters, same stream scratch) are
// replayed from a captured graph.  First sighting: plain launches (this also sizes the scratch planes).  Second:
// capture + instantiate + launch.  From then on: one cudaGraphLaunch.  Chains of fewer than three launches are not
// worth a graph; streams that are being captured by the caller, and the legacy default stream, launch directly.
int run_dev_cached(hgi_ctx* ctx, Scratch& sc, int mode, const uint8_t* src, uint32_t n_images, uint32_t w, uint32_t h,
                   uint32_t pitch, const hgi_params_t* prm, uint8_t* grid_out, uint8_t* recon_out, uint32_t* hist,
                   cudaStream_t st)
{
    const uint32_t levels = effective_levels(prm->levels, w, h);
    const bool multi = levels > (uint32_t)hgi::kMaxPassLevels;   // >= 3 launches
    auto plain = [&] {   // plain launches: the chain is not worth a graph, or its stream cannot be captured
        (void)cudaGetLastError();
        return run_dev(ctx, sc, mode, src, n_images, w, h, pitch, prm, grid_out, recon_out, hist, st);
    };
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (!multi || !graphs_enabled() || st == cudaStreamLegacy || st == cudaStreamPerThread ||
        cudaStreamIsCapturing(st, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone)
        return plain();
    ChainKey key{mode, prm->interp, prm->quant_kind, prm->quant_level, src, grid_out, recon_out, hist,
                 n_images, w, h, pitch, levels, &sc, sc.gen};
    ChainGraph* hit = nullptr;
    for (ChainGraph& g : ctx->chains)
        if (g.key == key) { hit = &g; break; }
    if (!hit) {   // first sighting: run it plainly and remember the key (the scratch generation may move: re-key after)
        const int rc = run_dev(ctx, sc, mode, src, n_images, w, h, pitch, prm, grid_out, recon_out, hist, st);
        if (rc) return rc;
        key.scratch_gen = sc.gen;
        for (size_t i = 0; i < ctx->chains.size();)   // chains that point into moved scratch planes are dead
            if (ctx->chains[i].key.scratch == &sc && ctx->chains[i].key.scratch_gen != sc.gen) {
                drop_chain(ctx->chains[i]);
                ctx->chains.erase(ctx->chains.begin() + (long)i);
            } else ++i;
        if (ctx->chains.size() >= kMaxChainGraphs) {
            size_t lru = 0;
            for (size_t i = 1; i < ctx->chains.size(); ++i)
                if (ctx->chains[i].last_use < ctx->chains[lru].last_use) lru = i;
            drop_chain(ctx->chains[lru]);
            ctx->chains.erase(ctx->chains.begin() + (long)lru);
        }
        ChainGraph g;
        g.key = key;
        g.last_use = ++ctx->chain_clock;
        ctx->chains.push_back(g);
        return HGI_OK;
    }
    hit->last_use = ++ctx->chain_clock;
    if (!hit->exec) {   // second sighting: capture the chain (nothing allocates now: the first run sized every buffer)
        const uint64_t before = hgi::launch_count();
        HGI_CUDA(ctx, cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        const int rc = run_dev(ctx, sc, mode, src, n_images, w, h, pitch, prm, grid_out, recon_out, hist, st);
        cudaGraph_t graph = nullptr;
        const cudaError_t ce = cudaStreamEndCapture(st, &graph);
        hit->launches = hgi::launch_count() - before;
        hgi::launch_count() = before;   // captured, not launched: the graph launch counts them
        cudaGraphExec_t exec = nullptr;
        if (rc == HGI_OK && ce == cudaSuccess && graph && sc.gen == key.scratch_gen &&
            cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess)
            hit->exec = exec;
        if (graph) cudaGraphDestroy(graph);
        if (rc != HGI_OK) {
            (void)cudaGetLastError();
            return rc;
        }
        if (!hit->exec) return plain();   // capture refused
    }
    HGI_CUDA(ctx, cudaGraphLaunch(hit->exec, st));
    hgi::launch_count() += hit->launches;
    ++ctx->graph_launches;
    return HGI_OK;
}

// Limits of the kernels' 32-bit offset arithmetic (tile-relative offsets up to 64 rows * pitch): rows shorter than 2^26
// bytes; the per-image residual histogram has 32-bit bins.
constexpr uint32_t kMaxPitch = 1u << 26;
// The residual histogram is one launch with at least one block per image, and a grid holds at most 2^31 - 1 blocks
// (its bins for that many images would take 2 TiB, more than any device has).
constexpr uint32_t kMaxHistImages = 0x7FFFFFFFu;

int cuda_rc(hgi_ctx* ctx, cudaError_t e) { return e == cudaSuccess ? HGI_OK : fail(ctx, e); }

// Two-slot pipeline of the reductions / colour conversion over host buffers (hgi_rgb_to_luma_u8, hgi_histogram_u8,
// hgi_error_metrics_u8): [0, n) is cut into chunks of `chunk` elements that alternate between slots 0 and 1, so the
// H2D copy of one chunk overlaps the kernel and the D2H copy of the other.  Each slot stages `in_per` (`out_per`) bytes
// per element of a chunk in `in` (`out`) and `hist_bytes` in `hist`.  enqueue(k, slot, off, len) puts one chunk's
// copies and kernel on slot k's stream; fold(k) takes in the result of slot k's last chunk once its stream has run
// it: before the slot is reused, and after the final drain.
template <class Enqueue, class Fold>
int run_chunks(hgi_ctx* ctx, size_t n, size_t chunk, size_t in_per, size_t out_per, size_t hist_bytes, Enqueue enqueue,
               Fold fold)
{
    const size_t cap = n < chunk ? n : chunk;
    const int ns = n > chunk ? 2 : 1;
    for (int k = 0; k < ns; ++k) {
        Slot& sl = ctx->slots[k];
        int rc = slot_stream(ctx, k);
        if (!rc) rc = reserve(ctx, sl.in, in_per * cap);
        if (!rc && out_per) rc = reserve(ctx, sl.out, out_per * cap);
        if (!rc && hist_bytes) rc = reserve(ctx, sl.hist, hist_bytes);
        if (rc) return rc;
    }
    bool pending[2] = {false, false};
    int rc = HGI_OK;
    size_t i = 0;
    for (size_t off = 0; off < n && !rc; off += chunk, ++i) {
        const int k = (int)(i & 1);
        Slot& sl = ctx->slots[k];
        if (pending[k]) {
            rc = cuda_rc(ctx, cudaStreamSynchronize(sl.stream));
            if (rc) break;
            fold(k);
            pending[k] = false;
        }
        rc = enqueue(k, sl, off, n - off < chunk ? n - off : chunk);
        if (!rc) pending[k] = true;
    }
    rc = drain(ctx, ns, rc);
    if (!rc)
        for (int k = 0; k < 2; ++k)
            if (pending[k]) fold(k);
    return rc;
}

constexpr int kEmptyJob = 1;   // check_job: the arguments are valid and there is nothing to do

// Argument checks of the encode / decode entry points, in this order: the handle, the parameters, the plane size
// (`size_ok`: a limit of the caller's own), an empty job (kEmptyJob, whatever its data pointers), null data pointers.
int check_job(bool handle, const hgi_params_t* prm, bool encode, uint32_t w, uint32_t h, uint32_t n_images,
              uint32_t pitch, std::initializer_list<const void*> ptrs, bool size_ok = true)
{
    if (!handle) return HGI_ERR_INVALID_ARG;
    if (int rc = check_params(prm, encode)) return rc;
    if (!size_ok || pitch < w || pitch >= kMaxPitch) return HGI_ERR_INVALID_ARG;
    if ((unsigned __int128)pitch * h * n_images >= ((unsigned __int128)1 << 62)) return HGI_ERR_INVALID_ARG;
    if ((size_t)w * h * n_images == 0) return kEmptyJob;
    for (const void* p : ptrs)
        if (!p) return HGI_ERR_INVALID_ARG;
    return HGI_OK;
}

// Host-pointer batch driver: images are cut into chunks that flow through `kSlots` stream slots
// (H2D -> kernels -> D2H), so copies in both directions overlap the kernels.
int run_host_chunks(hgi_ctx* ctx, int mode, const uint8_t* in, uint32_t n_images, uint32_t w, uint32_t h,
                    const hgi_params_t* prm, uint8_t* out, uint8_t* recon_out, uint32_t* hist_out, int* used_out)
{
    const size_t plane = (size_t)w * h;
    uint32_t per = (uint32_t)((ctx->chunk_bytes ? ctx->chunk_bytes : chunk_bytes()) / plane);
    if (per < 1) per = 1;
    if (per > n_images) per = n_images;
    const uint32_t n_chunks = (n_images + per - 1) / per;
    const int nslots = ctx->n_slots ? ctx->n_slots : slot_count();
    const int used = n_chunks < (uint32_t)nslots ? (int)n_chunks : nslots;
    for (int s = 0; s < used; ++s) {
        Slot& sl = ctx->slots[s];
        if (int rc = slot_stream(ctx, s)) return rc;
        *used_out = s + 1;
        int rc = reserve(ctx, sl.in, (size_t)per * plane);
        if (!rc) rc = reserve(ctx, sl.out, (size_t)per * plane);
        if (!rc && recon_out) rc = reserve(ctx, sl.aux, (size_t)per * plane);
        if (!rc && hist_out) rc = reserve(ctx, sl.hist, (size_t)per * 256 * sizeof(uint32_t));
        if (rc) return rc;
    }
    for (uint32_t c = 0; c < n_chunks; ++c) {
        Slot& sl = ctx->slots[c % (uint32_t)used];
        const uint32_t first = c * per;
        const uint32_t cnt = (n_images - first < per) ? n_images - first : per;
        const size_t off = (size_t)first * plane, bytes = (size_t)cnt * plane;
        // stream order on the slot protects its buffers and its scratch planes from the previous chunk that used them
        HGI_CUDA(ctx, cudaMemcpyAsync(sl.in.p, in + off, bytes, cudaMemcpyHostToDevice, sl.stream));
        uint8_t* d_grid = (mode == hgi::kModeEncode) ? sl.out.p : nullptr;
        uint8_t* d_recon = (mode == hgi::kModeEncode) ? (recon_out ? sl.aux.p : nullptr) : sl.out.p;
        uint32_t* d_hist = hist_out ? (uint32_t*)sl.hist.p : nullptr;
        int rc = run_dev(ctx, sl.scratch, mode, sl.in.p, cnt, w, h, w, prm, d_grid, d_recon, d_hist, sl.stream);
        if (rc) return rc;
        HGI_CUDA(ctx, cudaMemcpyAsync(out + off, sl.out.p, bytes, cudaMemcpyDeviceToHost, sl.stream));
        if (mode == hgi::kModeEncode && recon_out)
            HGI_CUDA(ctx, cudaMemcpyAsync(recon_out + off, sl.aux.p, bytes, cudaMemcpyDeviceToHost, sl.stream));
        if (hist_out)
            HGI_CUDA(ctx, cudaMemcpyAsync(hist_out + (size_t)first * 256, d_hist, (size_t)cnt * 256 * sizeof(uint32_t),
                                          cudaMemcpyDeviceToHost, sl.stream));
    }
    return HGI_OK;
}

// Host-pointer batch driver of one context: run_host_chunks, then every slot it used is drained.
int run_host(hgi_ctx* ctx, int mode, const uint8_t* in, uint32_t n_images, uint32_t w, uint32_t h,
             const hgi_params_t* prm, uint8_t* out, uint8_t* recon_out, uint32_t* hist_out)
{
    DeviceGuard g(ctx);
    if (!g.ok) return HGI_ERR_CUDA;
    int used = 0;
    const int rc = run_host_chunks(ctx, mode, in, n_images, w, h, prm, out, recon_out, hist_out, &used);
    return drain(ctx, used, rc);
}

// Window of a scalable decode (DESIGN.md "Scalable decode"): the region [u0, u1) of the scaled image is decoded from
// the window [x0, x1) with L' = max(L - k, 0) levels, x0 aligned down to S' = 2^L' (to max(S', 16) on the column axis:
// whole 16-byte chunks for the gather's 128-bit loads) and x1 = min(ws, floor((u1 - 1) / S') * S' + 2 S' + 1) -- the
// band rule y1 + S + 1 after aligning the end outwards to S'.  `r_out` receives the region (NULL: the scaled image).
int plan_region(uint32_t w, uint32_t h, uint32_t levels, uint32_t k, const hgi_rect_t* region, hgi_region_plan_t* p,
                hgi_rect_t* r_out)
{
    if (levels > HGI_MAX_LEVELS || k > HGI_MAX_LEVELS) return HGI_ERR_INVALID_ARG;
    const uint32_t ws = ceil_shift(w, k), hs = ceil_shift(h, k);
    const hgi_rect_t r = region ? *region : hgi_rect_t{0, 0, ws, hs};
    if (r.width == 0 || r.height == 0 || (uint64_t)r.x + r.width > ws || (uint64_t)r.y + r.height > hs)
        return HGI_ERR_INVALID_ARG;
    const uint32_t lp = levels > k ? levels - k : 0;
    const uint64_t S = 1ull << lp, A = S > 16 ? S : 16;
    auto end = [S](uint64_t u1, uint64_t n) {
        const uint64_t e = (u1 - 1) / S * S + 2 * S + 1;
        return e < n ? e : n;
    };
    const uint64_t x0 = r.x / A * A, y0 = r.y / S * S;
    const uint64_t x1 = end((uint64_t)r.x + r.width, ws), y1 = end((uint64_t)r.y + r.height, hs);
    *p = hgi_region_plan_t{ws, hs, lp, hgi_rect_t{(uint32_t)x0, (uint32_t)y0, (uint32_t)(x1 - x0), (uint32_t)(y1 - y0)},
                           (uint32_t)(r.x - x0), (uint32_t)(r.y - y0)};
    *r_out = r;
    return HGI_OK;
}

// Window of a batched crop (DESIGN.md "Batched crops"): hgi::crop_axis on each axis, so the window's extent depends on
// the crop's size only and every plane of a batch decodes a window of that extent.  `crop` is required.
int plan_crop(uint32_t w, uint32_t h, uint32_t levels, uint32_t k, const hgi_rect_t* crop, hgi_region_plan_t* p,
              hgi_rect_t* r_out)
{
    if (!crop) return HGI_ERR_INVALID_ARG;
    hgi_region_plan_t tight;
    hgi_rect_t r;
    if (int rc = plan_region(w, h, levels, k, crop, &tight, &r)) return rc;   // the same limits as a region
    const uint32_t lp = tight.levels;
    const hgi::CropAxis x = hgi::crop_axis(tight.scaled_width, r.width, lp, lp > 4 ? lp : 4, r.x);
    const hgi::CropAxis y = hgi::crop_axis(tight.scaled_height, r.height, lp, lp, r.y);
    *p = hgi_region_plan_t{tight.scaled_width, tight.scaled_height, lp, hgi_rect_t{x.start, y.start, x.extent, y.extent},
                           r.x - x.start, r.y - y.start};
    *r_out = r;
    return HGI_OK;
}

using PlanFn = int (*)(uint32_t, uint32_t, uint32_t, uint32_t, const hgi_rect_t*, hgi_region_plan_t*, hgi_rect_t*);

// Argument checks shared by the region and crop entry points: decode's, plus the rectangle (`plan`: its window rule).
int check_region(hgi_ctx* ctx, const hgi_params_t* prm, uint32_t w, uint32_t h, uint32_t n_images, uint32_t pitch,
                 uint32_t k, const hgi_rect_t* region, hgi_region_plan_t* pl, hgi_rect_t* r, PlanFn plan = plan_region)
{
    int rc = check_job(ctx, prm, false, w, h, n_images, pitch, {});
    if (rc < 0) return rc;   // an empty job is the region rules' to judge
    return plan(w, h, prm->levels, k, region, pl, r);
}

// Scalable decode of `n_images` planes: gather the window lattice (src + img * plane_stride + v * row_step + (u << k),
// see launch_region_gather) into dense planes, decode them on the tile path with L' levels, crop the region into
// d_out.  Launches plainly: region chains are not graph-cached.  With `crops.xy` every plane gathers and crops at its
// own origin (hgi::launch_region_gather); `pl` is then the uniform window of plan_crop, whose origin is not used.
int run_region(hgi_ctx* ctx, Scratch& sc, const uint8_t* src, uint64_t row_step, uint64_t plane_stride, bool vec,
               uint64_t row_avail, uint32_t k, uint32_t n_images, const hgi_region_plan_t& pl, const hgi_rect_t& r,
               const hgi_params_t* prm, uint8_t* d_out, uint32_t out_pitch, cudaStream_t st,
               const hgi::CropOrigins& crops = hgi::CropOrigins{})
{
    const uint32_t ww = pl.window.width, wh = pl.window.height, wpitch = align16(ww);
    const size_t bytes = (size_t)n_images * wpitch * wh;
    const uint32_t levels = effective_levels(pl.levels, ww, wh);   // 0: the window of the grid is the image
    int rc = reserve(ctx, sc, sc.region_in, bytes);
    if (!rc && levels) rc = reserve(ctx, sc, sc.region_out, bytes);
    if (rc) return rc;
    HGI_CUDA(ctx, hgi::launch_region_gather(src, row_step, plane_stride, k, ww, wh, wpitch, n_images, vec, row_avail,
                                            sc.region_in.p, st, crops));
    const uint8_t* win = sc.region_in.p;
    if (levels) {
        rc = run_tile_path(ctx, sc, hgi::kModeDecode, sc.region_in.p, n_images, ww, wh, wpitch, levels, prm, nullptr,
                           sc.region_out.p, st);
        if (rc) return rc;
        win = sc.region_out.p;
    }
    HGI_CUDA(ctx, hgi::launch_region_crop(win, wpitch, wh, pl.crop_x, pl.crop_y, r.width, r.height, n_images, d_out,
                                          out_pitch, st, crops));
    return HGI_OK;
}

}  // namespace

extern "C" {

int hgi_abi_version(void) { return HGI_ABI_VERSION; }

const char* hgi_strerror(int status)
{
    switch (status) {
        case HGI_OK: return "ok";
        case HGI_ERR_INVALID_ARG: return "invalid argument";
        case HGI_ERR_NO_DEVICE: return "no usable CUDA device (sm_100 required; there is no CPU fallback)";
        case HGI_ERR_CUDA: return "CUDA runtime error";
        case HGI_ERR_ALLOC: return "allocation failed";
        case HGI_ERR_BAD_MAGIC: return "incorrect magic number";
        case HGI_ERR_TRUNCATED: return "truncated or corrupt archive";
        case HGI_ERR_BUFFER_TOO_SMALL: return "output buffer too small";
        case HGI_ERR_UNSUPPORTED: return "unsupported option (no reference semantics)";
        default: return "unknown status";
    }
}

int hgi_ctx_create(int device, hgi_ctx_t** ctx_out)
{
    if (!ctx_out) return HGI_ERR_INVALID_ARG;
    *ctx_out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
        (void)cudaGetLastError();
        return HGI_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= count) return HGI_ERR_INVALID_ARG;
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return HGI_ERR_NO_DEVICE;
    if (prop.major != 10) return HGI_ERR_NO_DEVICE;  // kernels are built for sm_100a only
    if (!hgi::quant_swar_self_check()) return HGI_ERR_UNSUPPORTED;  // SWAR quantizer != reference table
    hgi_ctx* ctx = new (std::nothrow) hgi_ctx();
    if (!ctx) return HGI_ERR_ALLOC;
    ctx->device = device;
    {
        DeviceGuard g(ctx);
        cudaError_t e = g.ok ? cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) : ctx->last_err;
        if (e == cudaSuccess) e = cudaMalloc((void**)&ctx->d_metrics, 4 * sizeof(unsigned long long))   /* two per pipeline slot */;
        if (e == cudaSuccess) {
            *ctx_out = ctx;
            return HGI_OK;
        }
        if (ctx->stream) cudaStreamDestroy(ctx->stream);
        (void)cudaGetLastError();
    }
    delete ctx;   // after the guard, which writes to it when it ends
    return HGI_ERR_CUDA;
}

void hgi_ctx_destroy(hgi_ctx_t* ctx)
{
    if (!ctx) return;
    {
        DeviceGuard g(ctx);
        if (ctx->stream) cudaStreamSynchronize(ctx->stream);
        (void)cudaDeviceSynchronize();   // caller streams may still run chains that use the scratch sets
        for (ChainGraph& g : ctx->chains) drop_chain(g);
        ctx->chains.clear();
        for (StreamScratch* ss : ctx->caller_scratch) { free_scratch(ss->scratch); delete ss; }
        ctx->caller_scratch.clear();
        for (auto& s : ctx->slots) {
            free_scratch(s.scratch);
            if (s.stream) { cudaStreamSynchronize(s.stream); cudaStreamDestroy(s.stream); }
            free_bufs({&s.in, &s.out, &s.aux, &s.hist});
        }
        if (ctx->d_metrics) cudaFree(ctx->d_metrics);
        if (ctx->stream) cudaStreamDestroy(ctx->stream);
    }
    delete ctx;
}

int hgi_ctx_set_path(hgi_ctx_t* ctx, int path)
{
    // every path value runs the tile path (hgi.h): only the range is checked
    if (!ctx || path < HGI_PATH_TILE || path > HGI_PATH_TILE_TMA) return HGI_ERR_INVALID_ARG;
    return HGI_OK;
}

int hgi_ctx_set_pipeline(hgi_ctx_t* ctx, uint32_t chunk_mb, uint32_t slots)
{
    if (!ctx || chunk_mb > 4096 || slots > (uint32_t)kSlots) return HGI_ERR_INVALID_ARG;
    ctx->chunk_bytes = (size_t)chunk_mb << 20;
    ctx->n_slots = (int)slots;
    return HGI_OK;
}

int hgi_ctx_synchronize(hgi_ctx_t* ctx)
{
    if (!ctx) return HGI_ERR_INVALID_ARG;
    DeviceGuard g(ctx);
    if (!g.ok) return HGI_ERR_CUDA;
    HGI_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (auto& s : ctx->slots)
        if (s.stream) HGI_CUDA(ctx, cudaStreamSynchronize(s.stream));
    return HGI_OK;
}

int hgi_ctx_last_cuda_error(const hgi_ctx_t* ctx) { return ctx ? (int)ctx->last_err : 0; }
const char* hgi_ctx_last_cuda_error_string(const hgi_ctx_t* ctx)
{
    return ctx ? cudaGetErrorString(ctx->last_err) : "";
}
uint64_t hgi_ctx_kernel_launches(const hgi_ctx_t* ctx) { return ctx ? ctx->launches : 0; }
uint64_t hgi_ctx_graph_launches(const hgi_ctx_t* ctx) { return ctx ? ctx->graph_launches : 0; }

void* hgi_host_alloc(size_t bytes)
{
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    return p;
}

void hgi_host_free(void* ptr)
{
    if (ptr && cudaFreeHost(ptr) != cudaSuccess) (void)cudaGetLastError();
}

int hgi_host_register(void* ptr, size_t bytes)
{
    if (!ptr || !bytes) return HGI_ERR_INVALID_ARG;
    if (cudaHostRegister(ptr, bytes, cudaHostRegisterPortable) != cudaSuccess) {
        (void)cudaGetLastError();
        return HGI_ERR_CUDA;
    }
    return HGI_OK;
}

int hgi_host_unregister(void* ptr)
{
    if (!ptr) return HGI_ERR_INVALID_ARG;
    if (cudaHostUnregister(ptr) != cudaSuccess) {
        (void)cudaGetLastError();
        return HGI_ERR_CUDA;
    }
    return HGI_OK;
}

int hgi_quant_table(int quant_kind, int quant_level, uint8_t table_out[256], uint8_t* error_out)
{
    if (!table_out) return HGI_ERR_INVALID_ARG;
    if (quant_kind != HGI_QUANT_NOOP && quant_kind != HGI_QUANT_LINEAR) return HGI_ERR_INVALID_ARG;
    if (quant_kind == HGI_QUANT_LINEAR && (quant_level < 0 || quant_level > 3)) return HGI_ERR_INVALID_ARG;
    const uint32_t e = hgi::level_error(quant_kind, quant_level);
    for (uint32_t i = 0; i < 256; ++i) table_out[i] = (uint8_t)hgi::quant_entry(i, e);
    if (error_out) *error_out = (uint8_t)e;
    return HGI_OK;
}

int hgi_encode_dev_pitched(hgi_ctx_t* ctx, const uint8_t* d_images, uint32_t n_images, uint32_t width, uint32_t height,
                           uint32_t pitch, const hgi_params_t* params, uint8_t* d_grids_out, uint8_t* d_recon_out,
                           uint32_t* d_hist_out, void* stream)
{
    const bool bins_ok = !d_hist_out || ((uint64_t)width * height < (1ull << 32) && n_images <= kMaxHistImages);   // u32 bins
    if (int rc = check_job(ctx, params, true, width, height, n_images, pitch, {d_images, d_grids_out}, bins_ok))
        return rc == kEmptyJob ? HGI_OK : rc;
    DevCall dc(ctx, stream, true);
    if (dc.rc) return dc.rc;
    return run_dev_cached(ctx, *dc.sc, hgi::kModeEncode, d_images, n_images, width, height, pitch, params, d_grids_out,
                          d_recon_out, d_hist_out, dc.st);
}

int hgi_decode_dev_pitched(hgi_ctx_t* ctx, const uint8_t* d_grids, uint32_t n_images, uint32_t width, uint32_t height,
                           uint32_t pitch, const hgi_params_t* params, uint8_t* d_images_out, void* stream)
{
    if (int rc = check_job(ctx, params, false, width, height, n_images, pitch, {d_grids, d_images_out}))
        return rc == kEmptyJob ? HGI_OK : rc;
    DevCall dc(ctx, stream, true);
    if (dc.rc) return dc.rc;
    return run_dev_cached(ctx, *dc.sc, hgi::kModeDecode, d_grids, n_images, width, height, pitch, params, nullptr, d_images_out,
                          nullptr, dc.st);
}

int hgi_encode_dev(hgi_ctx_t* ctx, const uint8_t* d_images, uint32_t n_images, uint32_t width, uint32_t height,
                   const hgi_params_t* params, uint8_t* d_grids_out, uint8_t* d_recon_out, uint32_t* d_hist_out,
                   void* stream)
{
    return hgi_encode_dev_pitched(ctx, d_images, n_images, width, height, width, params, d_grids_out, d_recon_out, d_hist_out, stream);
}

int hgi_decode_dev(hgi_ctx_t* ctx, const uint8_t* d_grids, uint32_t n_images, uint32_t width, uint32_t height,
                   const hgi_params_t* params, uint8_t* d_images_out, void* stream)
{
    return hgi_decode_dev_pitched(ctx, d_grids, n_images, width, height, width, params, d_images_out, stream);
}

int hgi_histogram_dev(hgi_ctx_t* ctx, const uint8_t* d_grid, size_t n_per_image, uint32_t n_images,
                      uint32_t* d_hist_out, void* stream)
{
    if (!ctx || !d_hist_out) return HGI_ERR_INVALID_ARG;
    if (n_per_image >= ((size_t)1 << 32)) return HGI_ERR_INVALID_ARG;  // u32 bins
    if (n_images > kMaxHistImages) return HGI_ERR_INVALID_ARG;
    if (n_images == 0) return HGI_OK;
    if (!d_grid && n_per_image) return HGI_ERR_INVALID_ARG;
    DevCall dc(ctx, stream);
    if (dc.rc) return dc.rc;
    HGI_CUDA(ctx, hgi::launch_histogram(d_grid, (uint32_t)n_per_image, 1u, (uint32_t)n_per_image, n_images, d_hist_out, dc.st));
    return HGI_OK;
}

int hgi_rle_histogram_dev(hgi_ctx_t* ctx, const uint8_t* d_grid, size_t n, size_t block_bytes, size_t n_blocks,
                          uint32_t* d_hist_out, void* stream)
{
    if (!ctx || !d_hist_out || n_blocks == 0 || n_blocks > 65535) return HGI_ERR_INVALID_ARG;
    if (n && !d_grid) return HGI_ERR_INVALID_ARG;
    if (n_blocks == 1) block_bytes = n ? n : 1;
    if (block_bytes == 0 || block_bytes >= ((size_t)1 << 32) || (n_blocks > 1 && block_bytes % HGI_RLE_SEGMENT_BYTES != 0) ||
        (n_blocks - 1) * block_bytes > n || n_blocks * block_bytes < n)
        return HGI_ERR_INVALID_ARG;
    DevCall dc(ctx, stream);
    if (dc.rc) return dc.rc;
    HGI_CUDA(ctx, hgi::launch_rle_histogram(d_grid, n, block_bytes, (uint32_t)n_blocks, d_hist_out, dc.st));
    return HGI_OK;
}

int hgi_rle_histogram_u8(hgi_ctx_t* ctx, const uint8_t* grid, size_t n, size_t block_bytes, size_t n_blocks, uint32_t* hist_out)
{
    if (!ctx || !hist_out || n_blocks == 0 || n_blocks > 65535) return HGI_ERR_INVALID_ARG;
    if (n && !grid) return HGI_ERR_INVALID_ARG;
    DeviceGuard g(ctx);
    if (!g.ok) return HGI_ERR_CUDA;
    Slot& sl = ctx->slots[0];
    const size_t hbytes = n_blocks * HGI_RLE_TABLE_SYMBOLS * sizeof(uint32_t);
    int rc = slot_stream(ctx, 0);
    if (!rc) rc = reserve(ctx, sl.in, n ? n : 1);
    if (!rc) rc = reserve(ctx, sl.hist, hbytes);
    if (rc) return rc;
    if (n) HGI_CUDA(ctx, cudaMemcpyAsync(sl.in.p, grid, n, cudaMemcpyHostToDevice, sl.stream));
    rc = hgi_rle_histogram_dev(ctx, sl.in.p, n, block_bytes, n_blocks, (uint32_t*)sl.hist.p, sl.stream);
    if (rc == HGI_OK) rc = cuda_rc(ctx, cudaMemcpyAsync(hist_out, sl.hist.p, hbytes, cudaMemcpyDeviceToHost, sl.stream));
    return drain(ctx, 1, rc);
}

int hgi_error_metrics_dev(hgi_ctx_t* ctx, const uint8_t* d_before, const uint8_t* d_after, size_t n,
                          uint64_t* d_out, void* stream)
{
    if (!ctx || !d_out) return HGI_ERR_INVALID_ARG;
    if (n && (!d_before || !d_after)) return HGI_ERR_INVALID_ARG;
    DevCall dc(ctx, stream);
    if (dc.rc) return dc.rc;
    HGI_CUDA(ctx, hgi::launch_error_metrics(d_before, d_after, n, (unsigned long long*)d_out, dc.st));
    return HGI_OK;
}

int hgi_rgb_to_luma_dev(hgi_ctx_t* ctx, const uint8_t* d_rgb, size_t n_pixels, uint8_t* d_luma_out, void* stream)
{
    if (!ctx) return HGI_ERR_INVALID_ARG;
    if (n_pixels == 0) return HGI_OK;
    if (!d_rgb || !d_luma_out || n_pixels > ((size_t)1 << 60)) return HGI_ERR_INVALID_ARG;
    DevCall dc(ctx, stream);
    if (dc.rc) return dc.rc;
    HGI_CUDA(ctx, hgi::launch_rgb_to_luma(d_rgb, n_pixels, d_luma_out, dc.st));
    return HGI_OK;
}

int hgi_rgb_to_luma_u8(hgi_ctx_t* ctx, const uint8_t* rgb, size_t n_pixels, uint8_t* luma_out)
{
    if (!ctx) return HGI_ERR_INVALID_ARG;
    if (n_pixels == 0) return HGI_OK;
    if (!rgb || !luma_out || n_pixels > ((size_t)1 << 60)) return HGI_ERR_INVALID_ARG;
    DeviceGuard g(ctx);
    if (!g.ok) return HGI_ERR_CUDA;
    const size_t chunk = ctx->chunk_bytes ? ctx->chunk_bytes : ((size_t)64 << 20);   // pixels per chunk
    return run_chunks(ctx, n_pixels, chunk, 3, 1, 0, [&](int, Slot& sl, size_t off, size_t len) -> int {
        HGI_CUDA(ctx, cudaMemcpyAsync(sl.in.p, rgb + 3 * off, 3 * len, cudaMemcpyHostToDevice, sl.stream));
        HGI_CUDA(ctx, hgi::launch_rgb_to_luma(sl.in.p, len, sl.out.p, sl.stream));
        HGI_CUDA(ctx, cudaMemcpyAsync(luma_out + off, sl.out.p, len, cudaMemcpyDeviceToHost, sl.stream));
        return HGI_OK;
    }, [](int) {});
}

int hgi_encode_batch_u8(hgi_ctx_t* ctx, const uint8_t* images, uint32_t n_images, uint32_t width, uint32_t height,
                        const hgi_params_t* params, uint8_t* grids_out, uint32_t* hist_out)
{
    if (int rc = check_job(ctx, params, true, width, height, n_images, width, {images, grids_out}))
        return rc == kEmptyJob ? HGI_OK : rc;
    return run_host(ctx, hgi::kModeEncode, images, n_images, width, height, params, grids_out, nullptr, hist_out);
}

int hgi_decode_batch_u8(hgi_ctx_t* ctx, const uint8_t* grids, uint32_t n_images, uint32_t width, uint32_t height,
                        const hgi_params_t* params, uint8_t* images_out)
{
    if (int rc = check_job(ctx, params, false, width, height, n_images, width, {grids, images_out}))
        return rc == kEmptyJob ? HGI_OK : rc;
    return run_host(ctx, hgi::kModeDecode, grids, n_images, width, height, params, images_out, nullptr, nullptr);
}

int hgi_encode_u8(hgi_ctx_t* ctx, const uint8_t* image, uint32_t width, uint32_t height, const hgi_params_t* params,
                  uint8_t* grid_out, uint8_t* recon_out)
{
    if (int rc = check_job(ctx, params, true, width, height, 1, width, {image, grid_out}))
        return rc == kEmptyJob ? HGI_OK : rc;
    return run_host(ctx, hgi::kModeEncode, image, 1, width, height, params, grid_out, recon_out, nullptr);
}

int hgi_decode_u8(hgi_ctx_t* ctx, const uint8_t* grid, uint32_t width, uint32_t height, const hgi_params_t* params,
                  uint8_t* image_out)
{
    return hgi_decode_batch_u8(ctx, grid, 1, width, height, params, image_out);
}

int hgi_histogram_u8(hgi_ctx_t* ctx, const uint8_t* grid, size_t n, uint64_t hist_out[256])
{
    if (!ctx || !hist_out) return HGI_ERR_INVALID_ARG;
    for (int i = 0; i < 256; ++i) hist_out[i] = 0;
    if (n == 0) return HGI_OK;
    if (!grid) return HGI_ERR_INVALID_ARG;
    DeviceGuard g(ctx);
    if (!g.ok) return HGI_ERR_CUDA;
    // A chunk shorter than 2^32 bytes cannot overflow the u32 device bins and its length fits the launch's uint32_t;
    // the default stays far below that, a larger pipeline chunk (up to 4096 MiB) is cut to 4095 MiB.
    size_t chunk = ctx->chunk_bytes ? ctx->chunk_bytes : ((size_t)1 << 30);
    if (chunk > ((size_t)4095 << 20)) chunk = (size_t)4095 << 20;
    uint32_t part[2][256];
    return run_chunks(ctx, n, chunk, 1, 0, sizeof(part[0]), [&](int k, Slot& sl, size_t off, size_t len) -> int {
        HGI_CUDA(ctx, cudaMemcpyAsync(sl.in.p, grid + off, len, cudaMemcpyHostToDevice, sl.stream));
        HGI_CUDA(ctx, hgi::launch_histogram(sl.in.p, (uint32_t)len, 1u, (uint32_t)len, 1, (uint32_t*)sl.hist.p, sl.stream));
        HGI_CUDA(ctx, cudaMemcpyAsync(part[k], sl.hist.p, sizeof(part[k]), cudaMemcpyDeviceToHost, sl.stream));
        return HGI_OK;
    }, [&](int k) {
        for (int b = 0; b < 256; ++b) hist_out[b] += part[k][b];
    });
}

int hgi_error_metrics_u8(hgi_ctx_t* ctx, const uint8_t* before, const uint8_t* after, size_t n,
                         uint64_t* sum_sq_out, uint64_t* sd_int_out, uint32_t* max_abs_out)
{
    if (!ctx) return HGI_ERR_INVALID_ARG;
    if (n && (!before || !after)) return HGI_ERR_INVALID_ARG;
    unsigned long long total = 0, mx = 0;
    if (n) {
        DeviceGuard g(ctx);
        if (!g.ok) return HGI_ERR_CUDA;
        const size_t chunk = ctx->chunk_bytes ? ctx->chunk_bytes : ((size_t)256 << 20);
        unsigned long long part[2][2];
        const int rc = run_chunks(ctx, n, chunk, 1, 1, 0, [&](int k, Slot& sl, size_t off, size_t len) -> int {
            HGI_CUDA(ctx, cudaMemcpyAsync(sl.in.p, before + off, len, cudaMemcpyHostToDevice, sl.stream));
            HGI_CUDA(ctx, cudaMemcpyAsync(sl.out.p, after + off, len, cudaMemcpyHostToDevice, sl.stream));
            HGI_CUDA(ctx, hgi::launch_error_metrics(sl.in.p, sl.out.p, len, ctx->d_metrics + 2 * k, sl.stream));
            HGI_CUDA(ctx, cudaMemcpyAsync(part[k], ctx->d_metrics + 2 * k, sizeof(part[k]), cudaMemcpyDeviceToHost, sl.stream));
            return HGI_OK;
        }, [&](int k) {
            total += part[k][0];
            if (part[k][1] > mx) mx = part[k][1];
        });
        if (rc) return rc;
    }
    if (sum_sq_out) *sum_sq_out = total;
    if (sd_int_out) *sd_int_out = n ? total / n : 0;  // src/main.rs:106 integer division
    if (max_abs_out) *max_abs_out = (uint32_t)mx;
    return HGI_OK;
}


int hgi_plan_region(uint32_t width, uint32_t height, uint32_t levels, uint32_t scale_log2, const hgi_rect_t* region,
                    hgi_region_plan_t* plan_out)
{
    if (!plan_out) return HGI_ERR_INVALID_ARG;
    hgi_rect_t r;
    return plan_region(width, height, levels, scale_log2, region, plan_out, &r);
}

int hgi_decode_region_dev(hgi_ctx_t* ctx, const uint8_t* d_grids, uint32_t n_images, uint32_t width, uint32_t height,
                          uint32_t pitch, const hgi_params_t* params, uint32_t scale_log2, const hgi_rect_t* region,
                          uint8_t* d_out, uint32_t out_pitch, void* stream)
{
    hgi_region_plan_t pl;
    hgi_rect_t r;
    int rc = check_region(ctx, params, width, height, n_images, pitch, scale_log2, region, &pl, &r);
    if (rc) return rc;
    if (out_pitch < r.width) return HGI_ERR_INVALID_ARG;
    if (n_images == 0) return HGI_OK;
    if (!d_grids || !d_out) return HGI_ERR_INVALID_ARG;
    // the whole image into packed rows is a plain decode (with padded rows that one may write the padding)
    if (scale_log2 == 0 && r.width == width && r.height == height && out_pitch == pitch && pitch == width)
        return hgi_decode_dev_pitched(ctx, d_grids, n_images, width, height, pitch, params, d_out, stream);
    DevCall dc(ctx, stream, true);
    if (dc.rc) return dc.rc;
    const uint32_t k = scale_log2;
    const uint8_t* src = d_grids + ((size_t)pl.window.y << k) * pitch + ((size_t)pl.window.x << k);
    const uint64_t row_step = (uint64_t)pitch << k, plane_stride = (uint64_t)pitch * height;
    const bool vec = aligned16(src) && row_step % 16 == 0 && (n_images == 1 || plane_stride % 16 == 0);
    // the last row of the last plane ends at its pitch: no 128-bit load may reach past that
    const uint64_t row_avail = pitch - ((uint64_t)pl.window.x << k);
    return run_region(ctx, *dc.sc, src, row_step, plane_stride, vec, row_avail, k, n_images, pl, r, params, d_out, out_pitch,
                      dc.st);
}

int hgi_decode_region_u8(hgi_ctx_t* ctx, const uint8_t* grid, uint32_t width, uint32_t height, const hgi_params_t* params,
                         uint32_t scale_log2, const hgi_rect_t* region, uint8_t* image_out)
{
    hgi_region_plan_t pl;
    hgi_rect_t r;
    int rc = check_region(ctx, params, width, height, 1, width, scale_log2, region, &pl, &r);
    if (rc) return rc;
    if (!grid || !image_out) return HGI_ERR_INVALID_ARG;
    DeviceGuard g(ctx);
    if (!g.ok) return HGI_ERR_CUDA;
    const uint32_t k = scale_log2, ww = pl.window.width, wh = pl.window.height;
    // Stage the window's grid rows (every 2^k-th row, its column span) with one 2D copy.  Rows of the staging buffer
    // are readable up to (ww << k) bytes for k <= 3, so the gather's 128-bit loads never leave a row.
    const uint64_t span = ((uint64_t)(ww - 1) << k) + 1;
    const uint64_t spitch = ((k <= 3 ? (uint64_t)ww << k : span) + 15) & ~(uint64_t)15;
    const size_t out_bytes = (size_t)r.width * r.height;
    Slot& sl = ctx->slots[0];
    rc = slot_stream(ctx, 0);
    if (!rc) rc = reserve(ctx, sl.in, (size_t)spitch * wh);
    if (!rc) rc = reserve(ctx, sl.out, out_bytes);
    if (rc) return rc;
    const uint8_t* src = grid + ((size_t)pl.window.y << k) * width + ((size_t)pl.window.x << k);
    const size_t src_pitch = wh > 1 ? (size_t)width << k : (size_t)spitch;
    rc = cuda_rc(ctx, cudaMemcpy2DAsync(sl.in.p, spitch, src, src_pitch, span, wh, cudaMemcpyHostToDevice, sl.stream));
    if (!rc) rc = run_region(ctx, sl.scratch, sl.in.p, spitch, 0, true, spitch, k, 1, pl, r, params, sl.out.p, r.width, sl.stream);
    if (!rc) rc = cuda_rc(ctx, cudaMemcpyAsync(image_out, sl.out.p, out_bytes, cudaMemcpyDeviceToHost, sl.stream));
    return drain(ctx, 1, rc);
}

int hgi_plan_crop(uint32_t width, uint32_t height, uint32_t levels, uint32_t scale_log2, const hgi_rect_t* crop,
                  hgi_region_plan_t* plan_out)
{
    if (!plan_out) return HGI_ERR_INVALID_ARG;
    hgi_rect_t r;
    return plan_crop(width, height, levels, scale_log2, crop, plan_out, &r);
}

int hgi_decode_crops_dev(hgi_ctx_t* ctx, const uint8_t* d_grids, uint32_t n_images, uint32_t width, uint32_t height,
                         uint32_t pitch, const hgi_params_t* params, uint32_t scale_log2, uint32_t crop_width,
                         uint32_t crop_height, const int32_t* d_origins, uint8_t* d_out, uint32_t out_pitch, void* stream)
{
    hgi_region_plan_t pl;
    hgi_rect_t r;
    const hgi_rect_t crop{0, 0, crop_width, crop_height};
    int rc = check_region(ctx, params, width, height, n_images, pitch, scale_log2, &crop, &pl, &r, plan_crop);
    if (rc) return rc;
    if (out_pitch < crop_width) return HGI_ERR_INVALID_ARG;
    if (n_images == 0) return HGI_OK;
    if (!d_grids || !d_out || !d_origins || ((uintptr_t)d_origins & 3u)) return HGI_ERR_INVALID_ARG;
    DevCall dc(ctx, stream, true);
    if (dc.rc) return dc.rc;
    const uint32_t k = scale_log2;
    const uint64_t row_step = (uint64_t)pitch << k, plane_stride = (uint64_t)pitch * height;
    // each plane's window starts at a multiple of 16 bytes of its row (U0 << k, U0 a multiple of max(S', 16))
    const bool vec = aligned16(d_grids) && row_step % 16 == 0 && (n_images == 1 || plane_stride % 16 == 0);
    const hgi::CropOrigins crops{d_origins, pl.scaled_width, pl.scaled_height, crop_width, crop_height, pl.levels};
    return run_region(ctx, *dc.sc, d_grids, row_step, plane_stride, vec, pitch, k, n_images, pl, r, params, d_out, out_pitch,
                      dc.st, crops);
}

/* ---- pool: several GPUs behind one handle -------------------------------------------------------------------- */
}  // extern "C"

namespace {

// Contiguous [first, last) share of `rank` out of `world` (the first n % world ranks get one more).
void split_range(uint64_t n, uint32_t world, uint32_t rank, uint64_t* first, uint64_t* last)
{
    const uint64_t base = n / world, extra = n % world;
    *first = rank * base + (rank < extra ? rank : extra);
    *last = *first + base + (rank < extra ? 1 : 0);
}

// Bands of heights that are multiples of S = 2^levels; band [y0, y1) is bit-exact when computed from the input rows
// [y0, min(h, y1 + S + 1)): dependencies only point right/down (src/interpolator.rs:67-73), so the rows below a band
// are recomputed by its owner instead of being exchanged.  Empty bands are dropped.
int plan_bands(uint32_t height, uint32_t levels, uint32_t n_bands, hgi_band_t* out)
{
    const uint64_t S = 1ull << (levels > 31 ? 31 : levels);
    const uint64_t cells = (height + S - 1) / S;
    int n = 0;
    for (uint32_t r = 0; r < n_bands; ++r) {
        uint64_t c0, c1;
        split_range(cells, n_bands, r, &c0, &c1);
        const uint64_t y0 = c0 * S < height ? c0 * S : height, y1 = c1 * S < height ? c1 * S : height;
        if (y1 > y0) {
            const uint64_t in_y1 = y1 + S + 1 < height ? y1 + S + 1 : height;
            out[n++] = hgi_band_t{(uint32_t)y0, (uint32_t)y1, (uint32_t)in_y1};
        }
    }
    return n;
}

int pool_wait(hgi_pool* pool, int rc)
{
    for (size_t d = 0; d < pool->ctxs.size(); ++d) {
        DeviceGuard g(pool->ctxs[d]);
        rc = drain(pool->ctxs[d], pool->used[d], rc);
        pool->used[d] = 0;
    }
    return rc;
}

int pool_batch(hgi_pool* pool, int mode, const uint8_t* in, uint32_t n_images, uint32_t w, uint32_t h,
               const hgi_params_t* prm, uint8_t* out, uint32_t* hist_out)
{
    const size_t plane = (size_t)w * h;
    const uint32_t world = (uint32_t)pool->ctxs.size();
    int rc = HGI_OK;
    for (uint32_t d = 0; d < world && rc == HGI_OK; ++d) {
        uint64_t first, last;
        split_range(n_images, world, d, &first, &last);
        if (last == first) continue;
        hgi_ctx* ctx = pool->ctxs[d];
        DeviceGuard g(ctx);
        if (!g.ok) { rc = HGI_ERR_CUDA; break; }
        rc = run_host_chunks(ctx, mode, in + first * plane, (uint32_t)(last - first), w, h, prm, out + first * plane, nullptr,
                             hist_out ? hist_out + first * 256 : nullptr, &pool->used[d]);
    }
    return pool_wait(pool, rc);
}

// One band on one context, host pointers: rows [y0, in_y1) in, rows [y0, y1) out; enqueued on slot 0, not waited for.
int band_async(hgi_ctx* ctx, int mode, const uint8_t* in, uint32_t w, const hgi_band_t& b, const hgi_params_t* prm,
               uint8_t* out, int* used)
{
    Slot& sl = ctx->slots[0];
    int rc = slot_stream(ctx, 0);
    if (rc) return rc;
    *used = 1;
    const size_t rows_in = b.in_y1 - b.y0, rows_out = b.y1 - b.y0;
    rc = reserve(ctx, sl.in, rows_in * w);
    if (!rc) rc = reserve(ctx, sl.out, rows_in * w);
    if (rc) return rc;
    HGI_CUDA(ctx, cudaMemcpyAsync(sl.in.p, in + (size_t)b.y0 * w, rows_in * w, cudaMemcpyHostToDevice, sl.stream));
    rc = run_dev(ctx, sl.scratch, mode, sl.in.p, 1, w, (uint32_t)rows_in, w, prm, mode == hgi::kModeEncode ? sl.out.p : nullptr,
                 mode == hgi::kModeEncode ? nullptr : sl.out.p, nullptr, sl.stream);
    if (rc) return rc;
    HGI_CUDA(ctx, cudaMemcpyAsync(out + (size_t)b.y0 * w, sl.out.p, rows_out * w, cudaMemcpyDeviceToHost, sl.stream));
    return HGI_OK;
}

int pool_plane(hgi_pool* pool, int mode, const uint8_t* in, uint32_t w, uint32_t h, const hgi_params_t* prm, uint8_t* out)
{
    std::vector<hgi_band_t> bands(pool->ctxs.size());
    const int nb = plan_bands(h, prm->levels, (uint32_t)pool->ctxs.size(), bands.data());
    int rc = HGI_OK;
    for (int k = 0; k < nb && rc == HGI_OK; ++k) {
        hgi_ctx* ctx = pool->ctxs[(size_t)k];
        DeviceGuard g(ctx);
        if (!g.ok) { rc = HGI_ERR_CUDA; break; }
        rc = band_async(ctx, mode, in, w, bands[(size_t)k], prm, out, &pool->used[(size_t)k]);
    }
    return pool_wait(pool, rc);
}

int pool_bands_dev(hgi_pool* pool, int mode, const uint8_t* const* d_in, uint32_t w, uint32_t h, const hgi_params_t* prm,
                   uint8_t* const* d_out)
{
    std::vector<hgi_band_t> bands(pool->ctxs.size());
    const int nb = plan_bands(h, prm->levels, (uint32_t)pool->ctxs.size(), bands.data());
    for (int k = 0; k < nb; ++k) {
        if (!d_in[k] || !d_out[k]) return HGI_ERR_INVALID_ARG;
        hgi_ctx* ctx = pool->ctxs[(size_t)k];
        DevCall dc(ctx, nullptr, true);
        if (dc.rc) return dc.rc;
        const uint32_t rows_in = bands[(size_t)k].in_y1 - bands[(size_t)k].y0;
        const int rc = run_dev_cached(ctx, *dc.sc, mode, d_in[k], 1, w, rows_in, w, prm, mode == hgi::kModeEncode ? d_out[k] : nullptr,
                                      mode == hgi::kModeEncode ? nullptr : d_out[k], nullptr, dc.st);
        if (rc) return rc;
    }
    return HGI_OK;
}

}  // namespace

extern "C" {

int hgi_pool_create(const int* devices, int n_devices, hgi_pool_t** pool_out)
{
    if (!pool_out || n_devices < 0 || (n_devices > 0 && !devices)) return HGI_ERR_INVALID_ARG;
    *pool_out = nullptr;
    std::vector<int> devs;
    if (n_devices == 0) {   // every usable GPU of the box
        int count = 0;
        if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
            (void)cudaGetLastError();
            return HGI_ERR_NO_DEVICE;
        }
        for (int d = 0; d < count; ++d) {
            cudaDeviceProp prop{};
            if (cudaGetDeviceProperties(&prop, d) == cudaSuccess && prop.major == 10) devs.push_back(d);
        }
        if (devs.empty()) return HGI_ERR_NO_DEVICE;
    } else {
        devs.assign(devices, devices + n_devices);
    }
    hgi_pool* pool = new (std::nothrow) hgi_pool();
    if (!pool) return HGI_ERR_ALLOC;
    for (int d : devs) {
        hgi_ctx* ctx = nullptr;
        const int rc = hgi_ctx_create(d, &ctx);
        if (rc != HGI_OK) {
            for (hgi_ctx* c : pool->ctxs) hgi_ctx_destroy(c);
            delete pool;
            return rc;
        }
        pool->ctxs.push_back(ctx);
    }
    pool->used.assign(pool->ctxs.size(), 0);
    *pool_out = pool;
    return HGI_OK;
}

void hgi_pool_destroy(hgi_pool_t* pool)
{
    if (!pool) return;
    for (hgi_ctx* c : pool->ctxs) hgi_ctx_destroy(c);
    delete pool;
}

int hgi_pool_size(const hgi_pool_t* pool) { return pool ? (int)pool->ctxs.size() : 0; }

hgi_ctx_t* hgi_pool_ctx(hgi_pool_t* pool, int index)
{
    return (pool && index >= 0 && (size_t)index < pool->ctxs.size()) ? pool->ctxs[(size_t)index] : nullptr;
}

int hgi_pool_device(const hgi_pool_t* pool, int index)
{
    return (pool && index >= 0 && (size_t)index < pool->ctxs.size()) ? pool->ctxs[(size_t)index]->device : -1;
}

int hgi_pool_synchronize(hgi_pool_t* pool)
{
    if (!pool) return HGI_ERR_INVALID_ARG;
    int rc = HGI_OK;
    for (hgi_ctx* c : pool->ctxs) {
        const int r = hgi_ctx_synchronize(c);
        if (r != HGI_OK && rc == HGI_OK) rc = r;
    }
    return rc;
}

int hgi_pool_encode_batch_u8(hgi_pool_t* pool, const uint8_t* images, uint32_t n_images, uint32_t width, uint32_t height,
                             const hgi_params_t* params, uint8_t* grids_out, uint32_t* hist_out)
{
    if (int rc = check_job(pool, params, true, width, height, n_images, width, {images, grids_out}))
        return rc == kEmptyJob ? HGI_OK : rc;
    return pool_batch(pool, hgi::kModeEncode, images, n_images, width, height, params, grids_out, hist_out);
}

int hgi_pool_decode_batch_u8(hgi_pool_t* pool, const uint8_t* grids, uint32_t n_images, uint32_t width, uint32_t height,
                             const hgi_params_t* params, uint8_t* images_out)
{
    if (int rc = check_job(pool, params, false, width, height, n_images, width, {grids, images_out}))
        return rc == kEmptyJob ? HGI_OK : rc;
    return pool_batch(pool, hgi::kModeDecode, grids, n_images, width, height, params, images_out, nullptr);
}

int hgi_plan_bands(uint32_t height, uint32_t levels, uint32_t n_bands, hgi_band_t* bands_out, int* n_bands_out)
{
    if (!bands_out || !n_bands_out || levels > HGI_MAX_LEVELS || n_bands == 0) return HGI_ERR_INVALID_ARG;
    *n_bands_out = plan_bands(height, levels, n_bands, bands_out);
    return HGI_OK;
}

int hgi_pool_plan_bands(const hgi_pool_t* pool, uint32_t height, uint32_t levels, hgi_band_t* bands_out, int* n_bands_out)
{
    if (!pool || !bands_out || !n_bands_out || levels > HGI_MAX_LEVELS) return HGI_ERR_INVALID_ARG;
    *n_bands_out = plan_bands(height, levels, (uint32_t)pool->ctxs.size(), bands_out);
    return HGI_OK;
}

int hgi_pool_encode_plane_u8(hgi_pool_t* pool, const uint8_t* image, uint32_t width, uint32_t height,
                             const hgi_params_t* params, uint8_t* grid_out)
{
    if (int rc = check_job(pool, params, true, width, height, 1, width, {image, grid_out}))
        return rc == kEmptyJob ? HGI_OK : rc;
    return pool_plane(pool, hgi::kModeEncode, image, width, height, params, grid_out);
}

int hgi_pool_decode_plane_u8(hgi_pool_t* pool, const uint8_t* grid, uint32_t width, uint32_t height,
                             const hgi_params_t* params, uint8_t* image_out)
{
    if (int rc = check_job(pool, params, false, width, height, 1, width, {grid, image_out}))
        return rc == kEmptyJob ? HGI_OK : rc;
    return pool_plane(pool, hgi::kModeDecode, grid, width, height, params, image_out);
}

int hgi_pool_encode_bands_dev(hgi_pool_t* pool, const uint8_t* const* d_bands_in, uint32_t width, uint32_t height,
                              const hgi_params_t* params, uint8_t* const* d_bands_out)
{
    // the band arrays are checked with the handle, before the parameters
    if (int rc = check_job(pool && d_bands_in && d_bands_out, params, true, width, height, 1, width, {}))
        return rc == kEmptyJob ? HGI_OK : rc;
    return pool_bands_dev(pool, hgi::kModeEncode, d_bands_in, width, height, params, d_bands_out);
}

int hgi_pool_decode_bands_dev(hgi_pool_t* pool, const uint8_t* const* d_bands_in, uint32_t width, uint32_t height,
                              const hgi_params_t* params, uint8_t* const* d_bands_out)
{
    // the band arrays are checked with the handle, before the parameters
    if (int rc = check_job(pool && d_bands_in && d_bands_out, params, false, width, height, 1, width, {}))
        return rc == kEmptyJob ? HGI_OK : rc;
    return pool_bands_dev(pool, hgi::kModeDecode, d_bands_in, width, height, params, d_bands_out);
}

}  // extern "C"
