// hgi_region.cu -- the two copy kernels of scalable (reduced-resolution / region-of-interest) decode (DESIGN.md
// "Scalable decode"): gather a window of the 2^k lattice of the grid into dense planes, and crop the requested
// rectangle out of the decoded window planes.  The decode in between is the ordinary tile path.
#include <cstdint>

#include "hgi_kernels.h"

namespace hgi {

namespace {

constexpr uint32_t kCopyThreads = 256;

// Blocks of a grid-stride launch over `items` work items: enough to fill the 148 SMs, never more than the work.
uint32_t copy_blocks(uint64_t items)
{
    const uint64_t want = (items + kCopyThreads - 1) / kCopyThreads;
    return (uint32_t)(want < 148u * 16u ? want : 148u * 16u);
}

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) { return __byte_perm(a, b, sel); }

// Byte 0 of each of four words, packed little-endian.
__device__ __forceinline__ uint32_t low_bytes(uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
    return prmt(prmt(a, b, 0x0040u), prmt(c, d, 0x0040u), 0x5410u);
}

// Output chunk `c` (16 lattice points) of one window row from 128-bit loads of the source run: 16 << K bytes, i.e.
// 1, 2, 4 or 8 loads, compacted with PRMT.
template <int K>
__device__ __forceinline__ uint4 gather_vec(const uint8_t* __restrict__ srow, uint32_t c)
{
    const uint4* p = reinterpret_cast<const uint4*>(srow + ((size_t)c << (4 + K)));
    if constexpr (K == 0) {
        return __ldg(p);
    } else if constexpr (K == 1) {
        uint32_t o[4];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const uint4 v = __ldg(p + j);
            o[2 * j] = prmt(v.x, v.y, 0x6420u);
            o[2 * j + 1] = prmt(v.z, v.w, 0x6420u);
        }
        return make_uint4(o[0], o[1], o[2], o[3]);
    } else if constexpr (K == 2) {
        uint32_t o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint4 v = __ldg(p + j);
            o[j] = low_bytes(v.x, v.y, v.z, v.w);
        }
        return make_uint4(o[0], o[1], o[2], o[3]);
    } else {
        uint32_t o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint4 a = __ldg(p + 2 * j), b = __ldg(p + 2 * j + 1);
            o[j] = low_bytes(a.x, a.z, b.x, b.z);
        }
        return make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// Plane img of a crop batch: its origin (x, y) clamped into the scaled image, and the start (x0, y0) of its window.
struct CropWindow {
    uint32_t x, y, x0, y0;
};
__device__ __forceinline__ CropWindow crop_window(const CropOrigins& co, uint64_t img)
{
    const int32_t ox = __ldg(co.xy + 2 * img), oy = __ldg(co.xy + 2 * img + 1);   // 4-byte aligned only
    const uint32_t mx = co.ws - co.cw, my = co.hs - co.ch;
    const uint32_t x = ox < 0 ? 0u : ((uint32_t)ox > mx ? mx : (uint32_t)ox);
    const uint32_t y = oy < 0 ? 0u : ((uint32_t)oy > my ? my : (uint32_t)oy);
    const uint32_t ax = co.lp > 4u ? co.lp : 4u;
    return CropWindow{x, y, crop_axis(co.ws, co.cw, co.lp, ax, x).start, crop_axis(co.hs, co.ch, co.lp, co.lp, y).start};
}

// dst[img][v][u] = src[img * plane_stride + v * row_step + (u << k)] for u < ww, zero for ww <= u < dpitch.
// One thread writes 16 output bytes; a flat grid-stride loop over (window row, chunk) has no limit on the number of
// rows.  `vec`: the source rows are 16-byte aligned and readable for `row_avail` bytes, so chunks whose whole source
// run lies inside that take the 128-bit path (k <= 3); the others, and k >= 4 (one point per 16-byte chunk: a warp
// reads a contiguous run of every sector as in hgi_decimate_kernel), load point by point.  CROPS: plane img reads its
// own window, see launch_region_gather.
template <int K, bool CROPS>
__global__ void __launch_bounds__(kCopyThreads)
hgi_region_gather_kernel(const uint8_t* __restrict__ src, uint64_t row_step, uint64_t plane_stride, uint32_t kshift,
                         uint32_t ww, uint32_t wh, uint32_t dpitch, uint64_t n_rows, uint32_t vec, uint64_t row_avail,
                         uint8_t* __restrict__ dst, CropOrigins co)
{
    const uint32_t cpr = dpitch / 16u;
    const uint64_t total = n_rows * cpr;
    for (uint64_t it = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; it < total; it += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t row = it / cpr;
        const uint32_t c = (uint32_t)(it - row * cpr);
        const uint64_t img = row / wh, v = row - img * wh;
        const uint8_t* srow = src + img * plane_stride + v * row_step;
        uint64_t avail = row_avail;
        if constexpr (CROPS) {
            const CropWindow cw = crop_window(co, img);
            const uint64_t x0 = (uint64_t)cw.x0 << kshift;   // a multiple of 16: the start is aligned to max(S', 16)
            srow += cw.y0 * row_step + x0;
            avail -= x0;
        }
        uint4 out;
        if (K >= 0 && vec && 16u * c + 16u <= ww && ((uint64_t)(c + 1) << (4 + K)) <= avail) {
            out = gather_vec<K < 0 ? 0 : K>(srow, c);
        } else {
            uint32_t o[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (uint32_t i = 0; i < 16; ++i) {
                const uint32_t u = 16u * c + i;
                if (u < ww) o[i >> 2] |= (uint32_t)__ldg(srow + ((uint64_t)u << kshift)) << (8 * (i & 3));
            }
            out = make_uint4(o[0], o[1], o[2], o[3]);
        }
        *reinterpret_cast<uint4*>(dst + row * dpitch + 16u * c) = out;
    }
}

// out[img][r][j] = win[img][cy + r][cx + j] for r < rh, j < rw; output rows `out_pitch` bytes apart, planes
// out_pitch * rh.  Threads own 16-byte-aligned chunks of the output address space: whole chunks inside the
// rectangle row are one 128-bit store built from two aligned 128-bit loads of the window row (funnel shift by the
// misalignment); the chunks at the two ends of a row store byte by byte, so nothing outside the rectangle is written.
// CROPS: (cx, cy) is plane img's own, from its origin and window start.
template <bool CROPS>
__global__ void __launch_bounds__(kCopyThreads)
hgi_region_crop_kernel(const uint8_t* __restrict__ win, uint32_t wpitch, uint32_t wh, uint32_t cx, uint32_t cy,
                       uint32_t rw, uint32_t rh, uint64_t n_rows, uint8_t* __restrict__ out, uint32_t out_pitch,
                       CropOrigins co)
{
    const uint32_t cpr = (rw + 30u) / 16u + 1u;   // most chunks a row of rw bytes can touch
    const uint64_t total = n_rows * cpr;
    for (uint64_t it = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; it < total; it += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t row = it / cpr;
        const uint32_t c = (uint32_t)(it - row * cpr);
        const uint64_t img = row / rh, r = row - img * rh;
        uint8_t* drow = out + row * out_pitch;
        uint32_t ox = cx, oy = cy;
        if constexpr (CROPS) {
            const CropWindow cw = crop_window(co, img);
            ox = cw.x - cw.x0;
            oy = cw.y - cw.y0;
        }
        const uint8_t* srow = win + (img * wh + oy + r) * wpitch + ox;
        const int64_t j0 = 16 * (int64_t)c - (int64_t)((uintptr_t)drow & 15u);
        if (j0 >= (int64_t)rw) continue;
        if (j0 >= 0 && j0 + 16 <= (int64_t)rw) {
            const uint8_t* s = srow + j0;
            const uint32_t m = (uint32_t)((uintptr_t)s & 15u);
            const uint4* a = reinterpret_cast<const uint4*>(s - m);
            const uint4 lo = __ldg(a);
            const uint4 hi = m ? __ldg(a + 1) : make_uint4(0u, 0u, 0u, 0u);   // inside the row's 16-byte padding
            uint32_t w0 = lo.x, w1 = lo.y, w2 = lo.z, w3 = lo.w, w4 = hi.x, w5 = hi.y, w6 = hi.z, w7 = hi.w;
            if (m & 8u) { w0 = w2; w1 = w3; w2 = w4; w3 = w5; w4 = w6; w5 = w7; }
            if (m & 4u) { w0 = w1; w1 = w2; w2 = w3; w3 = w4; w4 = w5; }
            const uint32_t sh = 8u * (m & 3u);
            *reinterpret_cast<uint4*>(drow + j0) = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh),
                                                              __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int64_t j = j0 + i;
                if (j >= 0 && j < (int64_t)rw) drow[j] = __ldg(srow + j);
            }
        }
    }
}

template <bool CROPS>
void gather(const uint8_t* src, uint64_t row_step, uint64_t plane_stride, uint32_t k, uint32_t ww, uint32_t wh,
            uint32_t dpitch, uint64_t n_rows, bool vec, uint64_t row_avail, uint8_t* dst, cudaStream_t stream,
            const CropOrigins& co)
{
    const uint32_t nb = copy_blocks(n_rows * (dpitch / 16u));
    switch (k) {
        case 0: hgi_region_gather_kernel<0, CROPS><<<nb, kCopyThreads, 0, stream>>>(src, row_step, plane_stride, k, ww, wh, dpitch, n_rows, vec, row_avail, dst, co); break;
        case 1: hgi_region_gather_kernel<1, CROPS><<<nb, kCopyThreads, 0, stream>>>(src, row_step, plane_stride, k, ww, wh, dpitch, n_rows, vec, row_avail, dst, co); break;
        case 2: hgi_region_gather_kernel<2, CROPS><<<nb, kCopyThreads, 0, stream>>>(src, row_step, plane_stride, k, ww, wh, dpitch, n_rows, vec, row_avail, dst, co); break;
        case 3: hgi_region_gather_kernel<3, CROPS><<<nb, kCopyThreads, 0, stream>>>(src, row_step, plane_stride, k, ww, wh, dpitch, n_rows, vec, row_avail, dst, co); break;
        default: hgi_region_gather_kernel<-1, CROPS><<<nb, kCopyThreads, 0, stream>>>(src, row_step, plane_stride, k, ww, wh, dpitch, n_rows, 0u, 0u, dst, co); break;
    }
}

}  // namespace

cudaError_t launch_region_gather(const uint8_t* src, uint64_t row_step, uint64_t plane_stride, uint32_t k, uint32_t ww,
                                 uint32_t wh, uint32_t dpitch, uint32_t n_images, bool vec, uint64_t row_avail,
                                 uint8_t* dst, cudaStream_t stream, const CropOrigins& crops)
{
    if (ww == 0 || wh == 0 || n_images == 0) return cudaSuccess;
    const uint64_t n_rows = (uint64_t)n_images * wh;
    if (crops.xy) gather<true>(src, row_step, plane_stride, k, ww, wh, dpitch, n_rows, vec, row_avail, dst, stream, crops);
    else gather<false>(src, row_step, plane_stride, k, ww, wh, dpitch, n_rows, vec, row_avail, dst, stream, crops);
    ++launch_count();
    return cudaGetLastError();
}

cudaError_t launch_region_crop(const uint8_t* win, uint32_t wpitch, uint32_t wh, uint32_t cx, uint32_t cy, uint32_t rw,
                               uint32_t rh, uint32_t n_images, uint8_t* out, uint32_t out_pitch, cudaStream_t stream,
                               const CropOrigins& crops)
{
    if (rw == 0 || rh == 0 || n_images == 0) return cudaSuccess;
    const uint64_t n_rows = (uint64_t)n_images * rh;
    const uint32_t nb = copy_blocks(n_rows * ((rw + 30u) / 16u + 1u));
    if (crops.xy)
        hgi_region_crop_kernel<true><<<nb, kCopyThreads, 0, stream>>>(win, wpitch, wh, cx, cy, rw, rh, n_rows, out, out_pitch, crops);
    else
        hgi_region_crop_kernel<false><<<nb, kCopyThreads, 0, stream>>>(win, wpitch, wh, cx, cy, rw, rh, n_rows, out, out_pitch, crops);
    ++launch_count();
    return cudaGetLastError();
}

}  // namespace hgi
