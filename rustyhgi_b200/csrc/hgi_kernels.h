// hgi_kernels.h -- host-side launchers of the HGI CUDA kernels (internal to libhgi_b200.so).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace hgi {

// ---- fused tile path ----------------------------------------------------------------------
// One *pass* runs `nlev` (1..4) consecutive levels of the hierarchy for every tile of the
// lattice {(x,y) : x,y multiples of D = 2^d_log2}; see DESIGN.md "Pass decomposition".
constexpr int kTileW = 128;   // lattice points per tile row
constexpr int kTileH = 64;    // lattice rows per tile
constexpr int kTileThreads = 256;
constexpr int kMaxPassLevels = 4;

struct PassArgs {
    const uint8_t* src;      // encode: image planes; decode: grid planes (full resolution)
    uint8_t* grid_out;       // encode, D==1: grid planes
    uint8_t* recon_out;      // D==1: encode: optional reconstruction planes; decode: image planes
    const uint8_t* c_recon;  // compact reconstruction of the coarser pass (null => top pass)
    const uint8_t* c_q;      // compact symbols of the coarser pass (encode, non-top)
    uint8_t* s_recon;        // D>1: compact reconstruction written by this pass (wD x hD)
    uint8_t* s_q;            // D>1, encode: compact symbols written by this pass
    uint8_t* dec_in;         // D>1: scratch for the decimated source (this pass's lattice as a dense plane, pitch dpitch)
    uint32_t w, h;           // full-resolution plane size
    uint32_t pitch;          // bytes per row of src / grid_out / recon_out (>= w; == w for the reference's packed planes)
    uint32_t cpitch;         // bytes per row of c_recon / c_q
    uint32_t dpitch;         // D>1: bytes per row of s_recon / s_q / dec_in (16-byte multiple)
    uint32_t wD, hD;         // lattice size of this pass: ceil(w/D), ceil(h/D)
    uint32_t cw, ch;         // size of the coarser pass's compact planes
    uint32_t d_log2;         // log2(D)
    uint32_t nlev;           // levels fused in this pass (1..4); coarse step F = 2^nlev
    uint32_t tiles_x, tiles_y;
    uint32_t fast_tx, fast_itx, fast_ity;   // fast tile kernel: tiles per row, interior tile columns / rows (tile + halo inside the plane)
    uint32_t fast_rcol;                     // 1: there is exactly one non-interior tile column and it is a whole tile wide
    uint32_t n_images;
    // fast kernel, quantizing encode, interior tiles: L2 prefetch of the tile at pf_src = src + distance (the same tile of a later
    // plane, or a tile some tile rows further down a large plane) by the CTAs with image index < pf_zlim and tile row
    // < pf_ylim (the launcher's bounds for "the target tile exists and is interior"; pf_zlim = 0: off)
    uint32_t pf_zlim, pf_ylim;
    const uint8_t* pf_src;
    uint32_t quant_error;    // 0 => identity quantizer
    uint32_t vec_ok;         // rows and bases are 16-byte aligned => 128-bit global accesses (1: rows are whole chunks, 2: padded rows)
    // SWAR quantizer constants (quant_swar() of hgi_tile_swar.cuh, evaluated on the host per launch)
    uint32_t q_one, q_mul, q_add, q_shift, q_scale, q_rmask, q_qmul;
    uint32_t q_hK, q_hc1, q_hS, q_hc2;   // fp16x2 form
    // Split launches of the quantizing encode (interior / right tile columns / bottom tile rows) are independent of each
    // other: with a side stream and two events (owned by the caller's scratch set; all null = run them in sequence) the
    // two small edge launches run next to the interior launch instead of after it.
    cudaStream_t side_stream;
    cudaEvent_t ev_fork, ev_join;
};

// Dispatch of one pass.  kTileAuto: D == 1 passes on 16-byte-aligned planes go to the register-prefetch SWAR
// kernel (hgi_tile_fast.cu), everything else to the generic kernel (hgi_tile_kernels.cu).  kTileTma selects
// the persistent TMA-pipelined kernel (hgi_tile_tma.cu) for the eligible passes instead -- measured slower
// than the prefetch kernel in round 1 (profiles/), kept as a tested alternative.
enum TileVariant : int { kTileAuto = 0, kTileGeneric = 1, kTileTma = 2 };
// Kernels launched so far by the calling thread's launch_* calls (for hgi_ctx_kernel_launches).
uint64_t& launch_count();

cudaError_t launch_tile_pass(int mode, int interp, const PassArgs& args, cudaStream_t stream, int variant = kTileAuto);
cudaError_t launch_tile_pass_fast(int mode, int interp, const PassArgs& args, cudaStream_t stream);
cudaError_t launch_tile_pass_tma(int mode, int interp, const PassArgs& args, cudaStream_t stream, bool* used);
bool quant_swar_self_check();

// ---- per-level path -----------------------------------------------------------------------
struct LevelArgs {
    const uint8_t* grid_in;  // decode: residual planes
    uint8_t* grid_out;       // encode: residual planes
    uint8_t* recon;          // reconstruction planes, updated in place (encode: starts as image)
    uint32_t w, h;
    uint32_t step_log2;      // coarse step of this level = 2^step_log2 (sub-step = step/2)
    uint32_t n_images;
    uint32_t quant_error;
};
// D>1 passes of the SWAR kernels: gather the pass's lattice {multiples of 2^d_log2} of `n_images` pitched planes into
// dense planes (dpitch x hD each, zero padded), so that the pass itself runs on contiguous rows.
cudaError_t launch_decimate(const uint8_t* src, uint32_t pitch, uint32_t h, uint32_t d_log2, uint32_t wD, uint32_t hD,
                            uint32_t dpitch, uint32_t n_images, uint8_t* dst, cudaStream_t stream);
// Scalable decode (hgi_region.cu).  Gather: dst[img][v][u] = src[img * plane_stride + v * row_step + (u << k)] for the
// ww x wh window of `n_images` planes, rows of dst `dpitch` (16-byte multiple) apart, zero padded; `vec`: src, row_step
// and plane_stride are 16-byte aligned and every source row is readable for `row_avail` bytes (128-bit loads).
cudaError_t launch_region_gather(const uint8_t* src, uint64_t row_step, uint64_t plane_stride, uint32_t k, uint32_t ww,
                                 uint32_t wh, uint32_t dpitch, uint32_t n_images, bool vec, uint64_t row_avail,
                                 uint8_t* dst, cudaStream_t stream);
// Crop: out[img][r][j] = win[img][cy + r][cx + j] (window planes wpitch x wh) for the rw x rh rectangle; output rows
// out_pitch apart, planes out_pitch * rh apart; no byte outside the rectangle is written.
cudaError_t launch_region_crop(const uint8_t* win, uint32_t wpitch, uint32_t wh, uint32_t cx, uint32_t cy, uint32_t rw,
                               uint32_t rh, uint32_t n_images, uint8_t* out, uint32_t out_pitch, cudaStream_t stream);
cudaError_t launch_seed(int mode, const uint8_t* src, uint8_t* dst, uint32_t w, uint32_t h,
                        uint32_t levels, uint32_t n_images, cudaStream_t stream);
cudaError_t launch_level(int mode, int interp, const LevelArgs& args, cudaStream_t stream);

// ---- reductions ---------------------------------------------------------------------------
// `n_images` planes of `h` rows of `w` bytes, `pitch` bytes apart (pitch == w: one contiguous run of w * h bytes per
// image); hist_out[img][256] is overwritten.
cudaError_t launch_histogram(const uint8_t* data, uint32_t w, uint32_t h, uint32_t pitch, uint32_t n_images,
                             uint32_t* hist_out, cudaStream_t stream);
// Token frequencies of the run-length DEFLATE parse (286 literal/length symbols, rows of 288) of `n` contiguous bytes cut
// into blocks of `block_bytes` (the last one may be shorter): hist_out[n_blocks][288], overwritten.
cudaError_t launch_rle_histogram(const uint8_t* data, size_t n, size_t block_bytes, uint32_t n_blocks, uint32_t* hist_out,
                                 cudaStream_t stream);
cudaError_t launch_rgb_to_luma(const uint8_t* rgb, size_t n_pixels, uint8_t* luma, cudaStream_t stream);
cudaError_t launch_error_metrics(const uint8_t* before, const uint8_t* after, size_t n,
                                 unsigned long long* out2, cudaStream_t stream);

}  // namespace hgi
