// hgi_tile_kernels.cu -- generic (scalar, byte-wise) fused multi-level HGI tile kernel (sm_100a) + pass dispatch.
// The SWAR kernel (hgi_tile_fast.cu) shares this decomposition; this file keeps the plain
// formulation that the CPU model tests/tile_model.py mirrors line by line.
//
// One launch ("pass") runs up to four consecutive levels of the closed loop for every 128x64
// tile of the lattice {multiples of D}: the tile plus its right/bottom dependency halo is staged
// in shared memory once, all levels run there (coarse to fine, __syncthreads between levels,
// because each level predicts from the *reconstructed* coarser lattice), and the residual plane /
// reconstruction leaves with coalesced 128-bit stores.  HBM sees one read and one write per
// pixel per pass instead of one strided read-modify-write per level.
//
// Why a one-sided halo is enough: a new point of a cell reads only the cell's four corners, which
// lie at floor and floor+step (src/interpolator.rs:70-73), so dependencies only ever point
// right/down.  A tile therefore needs, beyond its own points, the lattice-s points up to
// X_s = TW-1, TW, TW+4, TW+8 for s = 1,2,4,8 and the coarse lattice (step F = 2^nlev) up to
// TW+F, which the previous pass (or the seeds) provides.  Halo points are recomputed, never
// exchanged; see DESIGN.md.
//
// Reference semantics: src/encoder.rs:39-71, src/decoder.rs:18-46, src/utils.rs:11-41,
// src/interpolator.rs:15-28,41-91, src/quantizator.rs:41-74 (restated in hgi_device.cuh).
#include "hgi_device.cuh"
#include "hgi_kernels.h"

namespace hgi {

namespace {

constexpr int TW = kTileW;
constexpr int TH = kTileH;
constexpr int NT = kTileThreads;
constexpr int FMAX = 1 << kMaxPassLevels;       // 16
constexpr int RPITCH = TW + 32;                 // 160: columns 0..TW+16 used, rows 16 B aligned
constexpr int RROWS = TH + FMAX + 1;            // rows 0..TH+16
constexpr int LOAD_CHUNKS = (TW + 16) / 16;     // 9 x 16 B per staged row (columns 0..TW+15)
constexpr int LOAD_ROWS = TH + 3;               // rows 0..TH-1, TH, TH+4, TH+8
constexpr int NWARPS = NT / 32;

__device__ __forceinline__ int staged_row(int idx) { return idx < TH ? idx : TH + 4 * (idx - TH); }

// Highest tile-relative coordinate at which a new point of sub-step s is still needed.
__device__ __forceinline__ int need_limit(int tile_extent, int s)
{
    return s == 1 ? tile_extent - 1 : (s == 2 ? tile_extent : tile_extent + s);
}

struct TileSmem {
    alignas(16) uint8_t R[RROWS * RPITCH];     // encode: pixels -> reconstruction; decode: residuals -> pixels
    alignas(16) uint8_t Q[TH * TW];            // encode: residual symbols of the tile
    uint8_t lut[256];
};

template <int MODE, int INTERP, bool IDENTITY>
__device__ __forceinline__ void process_cell(TileSmem& sm, int x0, int y0, int s, int xlim, int ylim,
                                             int xin, int yin, bool want_recon_finest)
{
    const int step = 2 * s;
    const uint32_t A = sm.R[y0 * RPITCH + x0];
    const uint32_t B = sm.R[(y0 + step) * RPITCH + x0];
    const uint32_t C = sm.R[y0 * RPITCH + x0 + step];
    const uint32_t D = sm.R[(y0 + step) * RPITCH + x0 + step];
    const uint32_t pred = predict<INTERP>(A, B, C, D);
    const int px[3] = {x0 + s, x0, x0 + s};
    const int py[3] = {y0, y0 + s, y0 + s};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int x = px[k], y = py[k];
        if (x > xlim || y > ylim || x >= xin || y >= yin) continue;
        uint8_t* r = &sm.R[y * RPITCH + x];
        if (MODE == kModeEncode) {
            uint32_t recon;
            const uint32_t q = encode_point<IDENTITY>(*r, pred, sm.lut, &recon);
            if (x < TW && y < TH) sm.Q[y * TW + x] = (uint8_t)q;
            if (s > 1 || want_recon_finest) *r = (uint8_t)recon;
        } else {
            *r = (uint8_t)((pred + *r) & 0xFFu);             // src/decoder.rs:39
        }
    }
}

template <int MODE, int INTERP, bool IDENTITY>
__global__ void __launch_bounds__(NT)
hgi_tile_kernel(const PassArgs p)
{
    __shared__ TileSmem sm;

    const int tid = threadIdx.x;
    const uint32_t tiles_per_image = p.tiles_x * p.tiles_y;
    const uint32_t img = blockIdx.x / tiles_per_image;
    const uint32_t t = blockIdx.x - img * tiles_per_image;
    const uint32_t ty = t / p.tiles_x, tx = t - ty * p.tiles_x;
    const int X0 = (int)(tx * TW), Y0 = (int)(ty * TH);       // lattice coordinates of the tile
    const int xin = (int)min((uint32_t)(TW + FMAX + 1), p.wD - (uint32_t)X0);  // in-image extent
    const int yin = (int)min((uint32_t)(TH + FMAX + 1), p.hD - (uint32_t)Y0);
    const size_t plane = (size_t)p.pitch * p.h;   // full-resolution planes: rows of p.pitch bytes
    const uint8_t* __restrict__ src = p.src + (size_t)img * plane;
    const bool top = (p.c_recon == nullptr);
    const int F = 1 << p.nlev;
    // 128-bit staging only for rows that are whole chunks (with padded rows a chunk may mix pixels and padding)
    const bool vec = p.vec_ok && (p.w & 15u) == 0;

    if (!IDENTITY) sm.lut[tid] = (uint8_t)quant_entry((uint32_t)tid, p.quant_error);

    // ---- stage the tile + halo ------------------------------------------------------------
    if (vec) {
        for (int it = tid; it < LOAD_ROWS * LOAD_CHUNKS; it += NT) {
            const int ri = it / LOAD_CHUNKS, c = it - ri * LOAD_CHUNKS;
            const int r = staged_row(ri);
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (r < yin && 16 * c < xin)
                v = __ldg(reinterpret_cast<const uint4*>(src + (size_t)(Y0 + r) * p.pitch + X0 + 16 * c));
            *reinterpret_cast<uint4*>(&sm.R[r * RPITCH + 16 * c]) = v;
        }
    } else {
        for (int it = tid; it < LOAD_ROWS * (TW + 16); it += NT) {
            const int ri = it / (TW + 16), x = it - ri * (TW + 16);
            const int r = staged_row(ri);
            uint8_t v = 0;
            if (r < yin && x < xin)
                v = __ldg(src + (((size_t)(Y0 + r)) << p.d_log2) * p.pitch + (((size_t)(X0 + x)) << p.d_log2));
            sm.R[r * RPITCH + x] = v;
        }
    }
    __syncthreads();

    // ---- coarse lattice of this pass: seeds (top pass) or the coarser pass's results --------
    {
        const int ncx = TW / F + 2, ncy = TH / F + 2;   // coarse points 0..TW+F / 0..TH+F
        for (int it = tid; it < ncx * ncy; it += NT) {
            const int cj = it / ncx, ci = it - cj * ncx;
            const int x = ci * F, y = cj * F;
            uint8_t rv = 0, qv = 0;
            if (x < xin && y < yin) {
                if (top) {
                    // src/encoder.rs:26-37 / src/decoder.rs:22-28: seed = the source byte itself
                    rv = __ldg(src + (((size_t)(Y0 + y)) << p.d_log2) * p.pitch + (((size_t)(X0 + x)) << p.d_log2));
                    qv = rv;
                } else {
                    const size_t co = ((size_t)img * p.ch + ((uint32_t)(Y0 + y) >> p.nlev)) * p.cpitch + ((uint32_t)(X0 + x) >> p.nlev);
                    rv = __ldg(p.c_recon + co);
                    if (MODE == kModeEncode) qv = __ldg(p.c_q + co);
                }
            }
            sm.R[y * RPITCH + x] = rv;
            if (MODE == kModeEncode && x < TW && y < TH) sm.Q[y * TW + x] = qv;
        }
    }
    __syncthreads();

    // ---- the closed loop: levels of this pass, coarse to fine --------------------------------
    const bool want_recon_finest = (p.d_log2 != 0) || (p.recon_out != nullptr);
    for (int s = F >> 1; s >= 1; s >>= 1) {
        const int step = 2 * s;
        const int xlim = need_limit(TW, s), ylim = need_limit(TH, s);
        const int ncx = TW / step + (s >= 2 ? 1 : 0), ncy = TH / step + (s >= 2 ? 1 : 0);
        for (int it = tid; it < ncx * ncy; it += NT) {
            const int cy = it / ncx, cx = it - cy * ncx;
            const int x0 = cx * step, y0 = cy * step;
            if (x0 >= xin || y0 >= yin) continue;
            process_cell<MODE, INTERP, IDENTITY>(sm, x0, y0, s, xlim, ylim, xin, yin, want_recon_finest);
        }
        __syncthreads();
    }

    // ---- write back --------------------------------------------------------------------------
    const int xout = min(TW, xin), yout = min(TH, yin);
    if (p.d_log2 == 0) {
        uint8_t* __restrict__ gout = (MODE == kModeEncode) ? p.grid_out + (size_t)img * plane : nullptr;
        uint8_t* __restrict__ rout = p.recon_out ? p.recon_out + (size_t)img * plane : nullptr;
        if (vec) {
            for (int it = tid; it < TH * (TW / 16); it += NT) {
                const int r = it / (TW / 16), c = it - r * (TW / 16);
                if (r >= yout || 16 * c >= xout) continue;
                const size_t off = (size_t)(Y0 + r) * p.pitch + X0 + 16 * c;
                if (MODE == kModeEncode)
                    *reinterpret_cast<uint4*>(gout + off) = *reinterpret_cast<const uint4*>(&sm.Q[r * TW + 16 * c]);
                if (rout)
                    *reinterpret_cast<uint4*>(rout + off) = *reinterpret_cast<const uint4*>(&sm.R[r * RPITCH + 16 * c]);
            }
        } else {
            for (int it = tid; it < TH * TW; it += NT) {
                const int r = it / TW, x = it - r * TW;
                if (r >= yout || x >= xout) continue;
                const size_t off = (size_t)(Y0 + r) * p.pitch + X0 + x;
                if (MODE == kModeEncode) gout[off] = sm.Q[r * TW + x];
                if (rout) rout[off] = sm.R[r * RPITCH + x];
            }
        }
    } else {
        // compact planes for the next (finer) pass
        const size_t cbase = (size_t)img * p.dpitch * p.hD;
        for (int it = tid; it < TH * TW; it += NT) {
            const int r = it / TW, x = it - r * TW;
            if (r >= yout || x >= xout) continue;
            const size_t off = cbase + (size_t)(Y0 + r) * p.dpitch + X0 + x;
            p.s_recon[off] = sm.R[r * RPITCH + x];
            if (MODE == kModeEncode) p.s_q[off] = sm.Q[r * TW + x];
        }
    }
}

template <int MODE, int INTERP>
cudaError_t launch_t(const PassArgs& a, cudaStream_t stream)
{
    const uint64_t nblocks = (uint64_t)a.tiles_x * a.tiles_y * a.n_images;
    if (nblocks == 0) return cudaSuccess;
    if (nblocks > 0x7FFFFFFFull) return cudaErrorInvalidConfiguration;
    if (MODE == kModeDecode || a.quant_error == 0)
        hgi_tile_kernel<MODE, INTERP, true><<<(uint32_t)nblocks, NT, 0, stream>>>(a);
    else
        hgi_tile_kernel<kModeEncode, INTERP, false><<<(uint32_t)nblocks, NT, 0, stream>>>(a);
    ++launch_count();
    return cudaGetLastError();
}

}  // namespace

uint64_t& launch_count()
{
    static thread_local uint64_t n = 0;
    return n;
}

cudaError_t launch_tile_pass(int mode, int interp, const PassArgs& a, cudaStream_t stream, bool generic)
{
    // the SWAR kernel takes any width / alignment and, through a decimated copy of the lattice, the D > 1 passes.
    // Only planes taller than 65535 tiles stay on the generic kernel
    if (!generic && (a.hD + 63) / 64 <= 65535u) return launch_tile_pass_fast(mode, interp, a, stream);
    if (mode == kModeEncode)
        return interp == kInterpLeftTop ? launch_t<kModeEncode, kInterpLeftTop>(a, stream)
                                        : launch_t<kModeEncode, kInterpCrossed>(a, stream);
    return interp == kInterpLeftTop ? launch_t<kModeDecode, kInterpLeftTop>(a, stream)
                                    : launch_t<kModeDecode, kInterpCrossed>(a, stream);
}

}  // namespace hgi
