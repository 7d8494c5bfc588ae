// hgi_level_kernels.cu -- per-level HGI kernels: one closed-loop pass over HBM per level.
//
// This is north_star's literal shape (seed kernel + one encode/decode kernel per level working
// on the planes in global memory).  The fused tile path (hgi_tile_kernels.cu) is the fast one;
// this path is kept as an independent CUDA formulation with identical results, selectable with
// hgi_ctx_set_path(ctx, HGI_PATH_PER_LEVEL).
//
// Reference: src/encoder.rs:26-37 / src/decoder.rs:22-28 (seed), src/encoder.rs:45-68 and
// src/decoder.rs:30-44 (level loop), src/utils.rs:11-41 (lattice), src/interpolator.rs:57-91.
#include "hgi_device.cuh"
#include "hgi_kernels.h"

namespace hgi {

// K0: dst[y][x] = src[y][x] for x,y multiples of 2^levels.
__global__ void __launch_bounds__(256)
hgi_seed_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, uint32_t w, uint32_t h,
                uint32_t levels, uint32_t sw, uint32_t sh, uint32_t n_images)
{
    const size_t plane = (size_t)w * h;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)sw * sh) return;
    const uint32_t sx = (uint32_t)(i % sw), sy = (uint32_t)(i / sw);
    for (uint32_t img = blockIdx.z; img < n_images; img += gridDim.z) {
        const size_t off = (size_t)img * plane + ((size_t)sy << levels) * w + ((size_t)sx << levels);
        dst[off] = src[off];
    }
}

// K1/K2: one thread per coarse cell; its (up to) three new points share one prediction.
template <int MODE, int INTERP, bool IDENTITY>
__global__ void __launch_bounds__(256)
hgi_level_kernel(LevelArgs a)
{
    __shared__ uint8_t lut[256];
    if (!IDENTITY) {
        for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x)
            lut[i] = (uint8_t)quant_entry(i, a.quant_error);
        __syncthreads();
    }
    const uint32_t step = 1u << a.step_log2, sub = step >> 1;
    const uint32_t cells_x = (a.w + step - 1) >> a.step_log2;
    const uint32_t cells_y = (a.h + step - 1) >> a.step_log2;
    const uint32_t cx = blockIdx.x * blockDim.x + threadIdx.x;
    if (cx >= cells_x) return;
    const size_t plane = (size_t)a.w * a.h;
    const uint32_t x0 = cx << a.step_log2, x1 = x0 + step;
    const bool xin = x1 < a.w;                               // src/interpolator.rs:77
    for (uint32_t img = blockIdx.z; img < a.n_images; img += gridDim.z) {
        uint8_t* __restrict__ R = a.recon + (size_t)img * plane;
        for (uint32_t cy = blockIdx.y; cy < cells_y; cy += gridDim.y) {
            const uint32_t y0 = cy << a.step_log2, y1 = y0 + step;
            const bool yin = y1 < a.h;
            const uint32_t A = R[(size_t)y0 * a.w + x0];
            const uint32_t B = yin ? R[(size_t)y1 * a.w + x0] : 0u;
            const uint32_t C = xin ? R[(size_t)y0 * a.w + x1] : 0u;
            const uint32_t D = (xin && yin) ? R[(size_t)y1 * a.w + x1] : 0u;
            const uint32_t pred = predict<INTERP>(A, B, C, D);

            const uint32_t px[3] = {x0 + sub, x0, x0 + sub};
            const uint32_t py[3] = {y0, y0 + sub, y0 + sub};
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                if (px[k] >= a.w || py[k] >= a.h) continue;
                const size_t off = (size_t)py[k] * a.w + px[k];
                if (MODE == kModeEncode) {
                    uint32_t recon;
                    const uint32_t q = encode_point<IDENTITY>(R[off], pred, lut, &recon);
                    a.grid_out[(size_t)img * plane + off] = (uint8_t)q;
                    R[off] = (uint8_t)recon;
                } else {
                    const uint32_t g = a.grid_in[(size_t)img * plane + off];
                    R[off] = (uint8_t)((pred + g) & 0xFFu);  // src/decoder.rs:39
                }
            }
        }
    }
}

cudaError_t launch_seed(int /*mode*/, const uint8_t* src, uint8_t* dst, uint32_t w, uint32_t h,
                        uint32_t levels, uint32_t n_images, cudaStream_t stream)
{
    const uint64_t S = 1ull << levels;
    const uint32_t sw = (uint32_t)((w + S - 1) / S), sh = (uint32_t)((h + S - 1) / S);
    if (sw == 0 || sh == 0 || n_images == 0) return cudaSuccess;
    dim3 grid((uint32_t)(((uint64_t)sw * sh + 255) / 256), 1, n_images < 65535u ? n_images : 65535u);
    hgi_seed_kernel<<<grid, 256, 0, stream>>>(src, dst, w, h, levels, sw, sh, n_images);
    ++launch_count();
    return cudaGetLastError();
}

template <int MODE, int INTERP>
static cudaError_t launch_level_t(const LevelArgs& a, cudaStream_t stream)
{
    const uint32_t step = 1u << a.step_log2;
    const uint32_t cells_x = (a.w + step - 1) >> a.step_log2;
    const uint32_t cells_y = (a.h + step - 1) >> a.step_log2;
    if (cells_x == 0 || cells_y == 0 || a.n_images == 0) return cudaSuccess;
    const uint32_t bx = cells_x >= 256 ? 256 : (cells_x >= 128 ? 128 : (cells_x >= 64 ? 64 : 32));
    dim3 block(bx, 1, 1);
    dim3 grid((cells_x + bx - 1) / bx, cells_y < 65535u ? cells_y : 65535u,
              a.n_images < 65535u ? a.n_images : 65535u);
    if (MODE == kModeDecode || a.quant_error == 0)
        hgi_level_kernel<MODE, INTERP, true><<<grid, block, 0, stream>>>(a);
    else
        hgi_level_kernel<kModeEncode, INTERP, false><<<grid, block, 0, stream>>>(a);
    ++launch_count();
    return cudaGetLastError();
}

cudaError_t launch_level(int mode, int interp, const LevelArgs& a, cudaStream_t stream)
{
    if (mode == kModeEncode)
        return interp == kInterpLeftTop ? launch_level_t<kModeEncode, kInterpLeftTop>(a, stream)
                                        : launch_level_t<kModeEncode, kInterpCrossed>(a, stream);
    return interp == kInterpLeftTop ? launch_level_t<kModeDecode, kInterpLeftTop>(a, stream)
                                    : launch_level_t<kModeDecode, kInterpCrossed>(a, stream);
}

}  // namespace hgi
