// hgi_reduce_kernels.cu -- residual histogram and `hgi test` error metrics (sm_100a).
//
// Histogram: north_star's "archive.rs residue histogram / frequency-table construction".  The
// reference has no such code (src/archive.rs:34-38 hands the bytes to flate2); the definition is
// hist[v] = #{grid bytes == v}.  Error metrics: src/main.rs:84-92 (sum of squared differences).
#include "hgi_device.cuh"
#include "hgi_kernels.h"

namespace hgi {

namespace {

#ifndef HGI_HIST_THREADS
#define HGI_HIST_THREADS 1024
#endif
#ifndef HGI_HIST_BLOCK_KB
#define HGI_HIST_BLOCK_KB 1024
#endif
constexpr int HT = HGI_HIST_THREADS;

// Residual histogram.  Each block owns a slice of one image (a contiguous byte range of a packed plane, a range of
// rows of a pitched one) and counts it into PRIVATE bins in shared memory: one column of 256 counters per lane,
// cell(bin, lane) at byte offset bin * 256 + lane * 4, so the 32 lanes of a warp always hit 32 different banks --
// every update is one conflict-free wavefront whatever the symbol statistics (a residual plane is mostly one symbol,
// the worst case for bins shared inside a warp: partially merged updates are 2.5x slower on this machine than
// conflict-free ones, and MATCH.ANY costs 67 clocks per warp, tools/ubench_hist.cu).  The 256-byte bin stride (half
// of it padding, 64 KB per block) makes the cell's offset ONE byte permute of the data word and the lane constant,
// [lane*4, byte k, 0, 0]: PRMT + base add + update per byte.  The warps of a block share the columns; the updates are
// fire-and-forget increments of the shared-memory unit (no value returns, no retry loop).  What decides the speed is
// how many warps keep that unit and the loads busy: 1024-thread blocks (two per SM, all 64 warp slots) with 1 MB of
// data each run at 5.8 TB/s, 256-thread blocks with 256 KB at 3.8 TB/s (A/B in profiles/r02_histogram.md).  At the
// end the block sums each bin over its 32 lanes with warp shuffles and issues one global RED per non-empty bin.
constexpr int kHistBinStride = 256;                         // bytes between bins
constexpr int kHistSmem = 256 * kHistBinStride;             // 64 KB
__device__ __forceinline__ void hist_count_word(uint8_t* bins, uint32_t w, uint32_t lane4)
{
    w ^= lane4 * 0x02020202u;   // row = bin ^ (8 * lane): equal symbols of different lanes go to different rows (see below)
    atomicAdd(reinterpret_cast<uint32_t*>(bins + __byte_perm(w, lane4, 0x6504u)), 1u);
    atomicAdd(reinterpret_cast<uint32_t*>(bins + __byte_perm(w, lane4, 0x6514u)), 1u);
    atomicAdd(reinterpret_cast<uint32_t*>(bins + __byte_perm(w, lane4, 0x6524u)), 1u);
    atomicAdd(reinterpret_cast<uint32_t*>(bins + __byte_perm(w, lane4, 0x6534u)), 1u);
}
__device__ __forceinline__ void hist_count_byte(uint8_t* bins, uint32_t b, uint32_t lane4)
{
    b ^= 2u * lane4;
    atomicAdd(reinterpret_cast<uint32_t*>(bins + b * kHistBinStride + lane4), 1u);
}

// one contiguous run of `len` bytes: byte head up to 16-byte alignment, 128-bit body (two loads in flight), byte tail
__device__ __forceinline__ void hist_count_run(const uint8_t* __restrict__ p, size_t len, uint8_t* bins, uint32_t lane4, int tid)
{
    size_t head = ((16 - ((uintptr_t)p & 15)) & 15);
    if (head > len) head = len;
    for (size_t i = tid; i < head; i += HT) hist_count_byte(bins, p[i], lane4);
    const size_t nvec = (len - head) / 16;
    const uint4* v4 = reinterpret_cast<const uint4*>(p + head);
    size_t i = tid;
    for (; i + HT < nvec; i += 2 * HT) {
        const uint4 v0 = __ldg(v4 + i), v1 = __ldg(v4 + i + HT);
        hist_count_word(bins, v0.x, lane4); hist_count_word(bins, v0.y, lane4); hist_count_word(bins, v0.z, lane4); hist_count_word(bins, v0.w, lane4);
        hist_count_word(bins, v1.x, lane4); hist_count_word(bins, v1.y, lane4); hist_count_word(bins, v1.z, lane4); hist_count_word(bins, v1.w, lane4);
    }
    for (; i < nvec; i += HT) {
        const uint4 v = __ldg(v4 + i);
        hist_count_word(bins, v.x, lane4); hist_count_word(bins, v.y, lane4); hist_count_word(bins, v.z, lane4); hist_count_word(bins, v.w, lane4);
    }
    for (size_t j = head + nvec * 16 + tid; j < len; j += HT) hist_count_byte(bins, p[j], lane4);
}

__global__ void __launch_bounds__(HT)
hgi_hist_kernel(const uint8_t* __restrict__ data, uint32_t w, uint32_t h, uint32_t pitch, uint32_t blocks_per_image,
                uint32_t* __restrict__ hist)
{
    extern __shared__ __align__(256) uint8_t bins[];   // kHistSmem bytes
    const int tid = threadIdx.x, lane = tid & 31;
    const uint32_t lane4 = 4u * (uint32_t)lane;
    for (int i = tid; i < 256 * 32; i += HT) *reinterpret_cast<uint32_t*>(bins + (i >> 5) * kHistBinStride + 4 * (i & 31)) = 0u;
    __syncthreads();
    const uint32_t img = blockIdx.x / blocks_per_image;
    const uint32_t b = blockIdx.x - img * blocks_per_image;
    const uint8_t* base = data + (size_t)img * pitch * h;
    if (pitch == w) {                               // packed plane: one run of w * h bytes, cut into 16-byte-aligned slices
        const size_t n = (size_t)w * h;
        const size_t per_block = ((n + blocks_per_image - 1) / blocks_per_image + 15) & ~(size_t)15;
        size_t lo = (size_t)b * per_block, hi = lo + per_block;
        if (hi > n) hi = n;
        if (lo < hi) hist_count_run(base + lo, hi - lo, bins, lane4, tid);
    } else {                                        // pitched plane: whole rows, the padding is not counted
        const uint32_t rows = (h + blocks_per_image - 1) / blocks_per_image;
        const uint32_t y0 = b * rows, y1 = y0 + rows < h ? y0 + rows : h;
        for (uint32_t y = y0; y < y1; ++y) hist_count_run(base + (size_t)y * pitch, w, bins, lane4, tid);
    }
    __syncthreads();
    // warp k reduces its share of the bins: lane-parallel reads of one bin row, shuffle tree
    constexpr int kBinsPerWarp = 256 / (HT / 32);
    for (int bin = (tid >> 5) * kBinsPerWarp; bin < (tid >> 5) * kBinsPerWarp + kBinsPerWarp; ++bin) {
        uint32_t v = *reinterpret_cast<const uint32_t*>(bins + (bin ^ (int)(2u * lane4)) * kHistBinStride + lane4);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
        if (lane == 0 && v) atomicAdd(&hist[(size_t)img * 256 + bin], v);
    }
}

// ---- token statistics of the run-length DEFLATE parse (entropy stage of the container, DESIGN.md 4.5) -----------
// The host writes a residual plane as DEFLATE literals plus distance-1 matches ("repeat the previous byte n times");
// on residual planes that is as small as zlib level 9.  This kernel builds the frequency table of that parse -- 286
// literal/length symbols -- so that the host only bit-packs.  The parse is fixed by hgi_rle_parse.h: the bytes of a
// block are cut into 512-byte segments; inside a segment every maximal run of equal bytes becomes one literal, then
// matches of min(258, rest) bytes while at least 3 bytes remain, then the last 0..2 bytes as literals.  One thread
// walks one segment; the counts go through a per-block table in shared memory (few updates per segment when the plane
// is made of runs, and updates of the same symbol by several lanes merge in the shared-memory increment unit).
constexpr int kRleSeg = 512;
constexpr int kRleSyms = 288;
__device__ __forceinline__ uint32_t rle_len_sym(uint32_t len)   // RFC 1951 3.2.5: length 3..258 -> symbol 257..285
{
    if (len == 258u) return 285u;
    const uint32_t l = len - 3u;
    const uint32_t e = l < 8u ? 0u : (uint32_t)(29 - __clz((int)l));   // floor(log2(l)) - 2 extra bits
    return 257u + 4u * e + (l >> e);
}

__global__ void __launch_bounds__(128)
hgi_rle_hist_kernel(const uint8_t* __restrict__ data, size_t n, size_t block_bytes, uint32_t* __restrict__ hist)
{
    __shared__ uint32_t bins[kRleSyms];
    for (int i = threadIdx.x; i < kRleSyms; i += blockDim.x) bins[i] = 0u;
    __syncthreads();
    const size_t blk = blockIdx.y;
    const size_t blo = blk * block_bytes, bhi = blo + block_bytes < n ? blo + block_bytes : n;
    const size_t seg = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t lo = blo + seg * kRleSeg;
    if (lo < bhi) {
        const size_t hi = lo + kRleSeg < bhi ? lo + kRleSeg : bhi;
        const uint8_t* p = data + lo;
        const uint32_t len = (uint32_t)(hi - lo);
        uint32_t i = 0;
        while (i < len) {
            const uint32_t b = p[i];
            uint32_t j = i + 1;
            while (j < len && p[j] == b) ++j;
            atomicAdd(&bins[b], 1u);
            uint32_t rem = j - i - 1u;
            while (rem >= 3u) {
                const uint32_t m = rem < 258u ? rem : 258u;
                atomicAdd(&bins[rle_len_sym(m)], 1u);
                rem -= m;
            }
            if (rem) atomicAdd(&bins[b], rem);
            i = j;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kRleSyms; i += blockDim.x)
        if (bins[i]) atomicAdd(&hist[blk * kRleSyms + i], bins[i]);
}

// 16 pixels per thread and iteration when both planes are 16-byte aligned: |a - b| per byte, squares summed with a
// 4-way dot product (exact: 4 * 255^2 per word fits 32 bits, widened to 64 bits per 16 bytes), running byte-wise max.
__global__ void __launch_bounds__(256)
hgi_error_kernel(const uint8_t* __restrict__ before, const uint8_t* __restrict__ after, size_t n,
                 unsigned long long* __restrict__ out2, int vec_ok)
{
    unsigned long long sum = 0;
    uint32_t mx = 0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t groups = vec_ok ? n / 16 : 0;
    uint32_t mx4 = 0;
    for (size_t g = tid; g < groups; g += stride) {
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(before) + g);
        const uint4 b = __ldg(reinterpret_cast<const uint4*>(after) + g);
        const uint32_t d0 = __vabsdiffu4(a.x, b.x), d1 = __vabsdiffu4(a.y, b.y);   // src/main.rs:89
        const uint32_t d2 = __vabsdiffu4(a.z, b.z), d3 = __vabsdiffu4(a.w, b.w);
        mx4 = __vmaxu4(__vmaxu4(mx4, d0), __vmaxu4(d1, __vmaxu4(d2, d3)));
        sum += __dp4a(d0, d0, __dp4a(d1, d1, __dp4a(d2, d2, __dp4a(d3, d3, 0u))));   // src/main.rs:91
    }
    mx = max(max(mx4 & 255u, (mx4 >> 8) & 255u), max((mx4 >> 16) & 255u, mx4 >> 24));
    for (size_t i = groups * 16 + tid; i < n; i += stride) {
        const int d = (int)before[i] - (int)after[i];        // src/main.rs:89
        const uint32_t a = (uint32_t)(d < 0 ? -d : d);
        mx = max(mx, a);
        sum += (unsigned long long)(a * a);                  // src/main.rs:91
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sum += __shfl_xor_sync(0xFFFFFFFFu, sum, o);
        mx = max(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, o));
    }
    __shared__ unsigned long long ssum[8];
    __shared__ uint32_t smx[8];
    if ((threadIdx.x & 31) == 0) { ssum[threadIdx.x >> 5] = sum; smx[threadIdx.x >> 5] = mx; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) { sum += ssum[w]; mx = max(mx, smx[w]); }
        atomicAdd(&out2[0], sum);
        atomicMax(&out2[1], (unsigned long long)mx);
    }
}

// RGB -> luma, the `image` 0.19 `to_luma()` that src/main.rs:42,74 calls before encoding (SURVEY.md 8 f-2):
// l = 0.2126f*r + 0.7152f*g + 0.0722f*b in f32, evaluated left to right with separately rounded
// multiplies and adds (Rust never contracts to FMA), truncated to u8.  __fmul_rn/__fadd_rn are never
// fused by nvcc, independent of -fmad.
__device__ __forceinline__ uint32_t luma_of(uint32_t r, uint32_t g, uint32_t b)
{
    float l = __fmul_rn(0.2126f, (float)r);
    l = __fadd_rn(l, __fmul_rn(0.7152f, (float)g));
    l = __fadd_rn(l, __fmul_rn(0.0722f, (float)b));
    return (uint32_t)l;   // truncation; l < 256
}

// The same arithmetic without the conversion unit: byte `k` of word `w` becomes the float 2^23 + byte by a single
// PRMT into the mantissa of 0x4B000000, minus 2^23 gives (float)byte exactly; the truncation is an add of 2^23
// rounded toward zero, whose low mantissa byte is floor(l) (0 <= l < 256).  Returns that float's bits.
__device__ __forceinline__ float byte_to_f32(uint32_t w, uint32_t k)
{
    return __fadd_rn(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540u + k)), -8388608.0f);
}
__device__ __forceinline__ uint32_t luma_bits(float r, float g, float b)
{
    float l = __fmul_rn(0.2126f, r);
    l = __fadd_rn(l, __fmul_rn(0.7152f, g));
    l = __fadd_rn(l, __fmul_rn(0.0722f, b));
    return __float_as_uint(__fadd_rz(l, 8388608.0f));   // low byte = (u8)l
}

// 16 pixels per thread: three 128-bit loads (48 RGB bytes), one 128-bit store.
__global__ void __launch_bounds__(256)
hgi_luma_kernel(const uint8_t* __restrict__ rgb, size_t n_pixels, uint8_t* __restrict__ luma, int vec_ok)
{
    const size_t groups = n_pixels / 16;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (vec_ok) {
        for (size_t gidx = tid; gidx < groups; gidx += stride) {
            const uint4* src = reinterpret_cast<const uint4*>(rgb + gidx * 48);
            const uint4 v0 = __ldg(src), v1 = __ldg(src + 1), v2 = __ldg(src + 2);
            const uint32_t w[12] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w};
            uint32_t out[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {   // 4 pixels = 12 bytes = words 3q..3q+2
                const uint32_t a = w[3 * q], b = w[3 * q + 1], c = w[3 * q + 2];
                const uint32_t l0 = luma_bits(byte_to_f32(a, 0), byte_to_f32(a, 1), byte_to_f32(a, 2));
                const uint32_t l1 = luma_bits(byte_to_f32(a, 3), byte_to_f32(b, 0), byte_to_f32(b, 1));
                const uint32_t l2 = luma_bits(byte_to_f32(b, 2), byte_to_f32(b, 3), byte_to_f32(c, 0));
                const uint32_t l3 = luma_bits(byte_to_f32(c, 1), byte_to_f32(c, 2), byte_to_f32(c, 3));
                out[q] = __byte_perm(__byte_perm(l0, l1, 0x0040u), __byte_perm(l2, l3, 0x0040u), 0x5410u);
            }
            *reinterpret_cast<uint4*>(luma + gidx * 16) = make_uint4(out[0], out[1], out[2], out[3]);
        }
    }
    const size_t first = vec_ok ? groups * 16 : 0;
    for (size_t i = first + tid; i < n_pixels; i += stride)
        luma[i] = (uint8_t)luma_of(rgb[3 * i], rgb[3 * i + 1], rgb[3 * i + 2]);
}

}  // namespace

cudaError_t launch_rgb_to_luma(const uint8_t* rgb, size_t n_pixels, uint8_t* luma, cudaStream_t stream)
{
    if (n_pixels == 0) return cudaSuccess;
    const int vec_ok = (((uintptr_t)rgb | (uintptr_t)luma) & 15u) == 0;
    uint64_t blocks = (n_pixels / 16 + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > 148 * 32) blocks = 148 * 32;
    hgi_luma_kernel<<<(uint32_t)blocks, 256, 0, stream>>>(rgb, n_pixels, luma, vec_ok);
    ++launch_count();
    return cudaGetLastError();
}

cudaError_t launch_histogram(const uint8_t* data, uint32_t w, uint32_t h, uint32_t pitch, uint32_t n_images,
                             uint32_t* hist_out, cudaStream_t stream)
{
    if (n_images == 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(hist_out, 0, (size_t)n_images * 256 * sizeof(uint32_t), stream);
    const uint64_t n_per_image = (uint64_t)w * h;
    if (e != cudaSuccess || n_per_image == 0) return e;
    // Zeroing and reducing the 32 KB of counters costs a block about as much as counting 32 KB of data: a block gets
    // 1 MiB when the job is large; smaller jobs are cut so that every SM still has blocks (not below 64 KiB)
    {   // function attributes are per device: opt in to 64 KB of dynamic shared memory once on each
        static bool done[64] = {};
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return cudaGetLastError();
        if (dev < 0 || dev >= 64 || !done[dev]) {
            e = cudaFuncSetAttribute(hgi_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kHistSmem);
            if (e != cudaSuccess) return e;
            if (dev >= 0 && dev < 64) done[dev] = true;
        }
    }
    const uint64_t total = n_per_image * n_images;
    uint64_t per_block = ((total / 592 + 16383) / 16384) * 16384;            // ~4 blocks per SM
    if (per_block < (64u << 10)) per_block = 64u << 10;
    if (per_block > ((uint64_t)HGI_HIST_BLOCK_KB << 10)) per_block = (uint64_t)HGI_HIST_BLOCK_KB << 10;
    uint64_t bpi = (n_per_image + per_block - 1) / per_block;
    if (bpi < 1) bpi = 1;
    if (pitch != w && bpi > h) bpi = h;
    if (bpi * n_images > 0x7FFFFFFFull) bpi = 0x7FFFFFFFull / n_images;
    if (bpi < 1) return cudaErrorInvalidConfiguration;
    hgi_hist_kernel<<<(uint32_t)(bpi * n_images), HT, kHistSmem, stream>>>(data, w, h, pitch, (uint32_t)bpi, hist_out);
    ++launch_count();
    return cudaGetLastError();
}

cudaError_t launch_rle_histogram(const uint8_t* data, size_t n, size_t block_bytes, uint32_t n_blocks, uint32_t* hist_out,
                                 cudaStream_t stream)
{
    if (n_blocks == 0) return cudaSuccess;
    cudaError_t e = cudaMemsetAsync(hist_out, 0, (size_t)n_blocks * kRleSyms * sizeof(uint32_t), stream);
    if (e != cudaSuccess || n == 0) return e;
    const size_t segs = (block_bytes + kRleSeg - 1) / kRleSeg;
    const size_t gx = (segs + 127) / 128;
    if (gx > 0x7FFFFFFFull || n_blocks > 65535u) return cudaErrorInvalidConfiguration;
    hgi_rle_hist_kernel<<<dim3((uint32_t)gx, n_blocks), 128, 0, stream>>>(data, n, block_bytes, hist_out);
    ++launch_count();
    return cudaGetLastError();
}

cudaError_t launch_error_metrics(const uint8_t* before, const uint8_t* after, size_t n,
                                 unsigned long long* out2, cudaStream_t stream)
{
    cudaError_t e = cudaMemsetAsync(out2, 0, 2 * sizeof(unsigned long long), stream);
    if (e != cudaSuccess || n == 0) return e;
    const int vec_ok = (((uintptr_t)before | (uintptr_t)after) & 15u) == 0;
    uint64_t blocks = (n + 256 * 64 - 1) / (256 * 64);
    if (blocks > 148 * 16) blocks = 148 * 16;
    hgi_error_kernel<<<(uint32_t)blocks, 256, 0, stream>>>(before, after, n, out2, vec_ok);
    ++launch_count();
    return cudaGetLastError();
}

}  // namespace hgi
