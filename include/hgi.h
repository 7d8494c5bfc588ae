/*
 * hgi.h -- C ABI of libhgi_b200.so: the B200-native implementation of RustyHGI's
 * hierarchical-grid encode/decode loop.
 *
 * This header is the drop-in boundary for that path.  The reference (Rust crate `hgi`) has no
 * FFI of its own -- its public surface is the generic `Encoder<I,Q>` / `Decoder<I>` pair plus
 * the `Quantizator`/`Interpolator` option types re-exported at src/lib.rs:16-23 -- so each entry
 * point below cites the reference item it replaces (file:line relative to the reference tree).
 * INTEGRATION.md shows the `extern "C"` block + safe wrappers a maintainer would add on the Rust
 * side; include/hgi.hpp is the same mirror in C++.
 *
 * Conventions
 *  - Planes are row-major u8 with stride == width, exactly `image::GrayImage` / `Grid::buffer`
 *    (src/grid.rs:19-27).  A batch is `n_images` such planes back to back.
 *  - Every function returns HGI_OK (0) or a negative hgi_status_t; nothing aborts or throws.
 *  - `*_u8` entry points take HOST pointers (the reference-facing calls; copies are inside).
 *    `*_dev` entry points take DEVICE pointers and enqueue on `stream` (a cudaStream_t passed as
 *    void*; NULL = the context's own stream) without synchronising.
 *  - A context is bound to one CUDA device; calls on one context are stream-ordered and must not
 *    be issued concurrently from several host threads.  Distinct contexts are independent.
 *    `*_dev` calls on different streams of one context may overlap on the device: each stream
 *    gets its own scratch planes (the 32 most recently used streams are kept).
 *  - There is no CPU fallback: if no CUDA device is usable, hgi_ctx_create fails.
 */
#ifndef HGI_H_
#define HGI_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HGI_ABI_VERSION 2

typedef struct hgi_ctx hgi_ctx_t;

/* Status codes. */
typedef enum {
    HGI_OK = 0,
    HGI_ERR_INVALID_ARG = -1,   /* null pointer, levels > HGI_MAX_LEVELS, bad enum, w*h overflow */
    HGI_ERR_NO_DEVICE = -2,     /* no usable CUDA device / wrong architecture */
    HGI_ERR_CUDA = -3,          /* a CUDA runtime call failed; see hgi_ctx_last_cuda_error */
    HGI_ERR_ALLOC = -4,         /* host or device allocation failed */
    HGI_ERR_BAD_MAGIC = -5,     /* archive: "incorrect magic number" (src/archive.rs:47-50) */
    HGI_ERR_TRUNCATED = -6,     /* archive: short read / corrupt deflate stream */
    HGI_ERR_BUFFER_TOO_SMALL = -7,
    HGI_ERR_UNSUPPORTED = -8    /* e.g. interpolation tag with no reference semantics */
} hgi_status_t;

/* src/interpolator.rs:4-9 `InterpolationType` (values = bincode variant indices).  Only Crossed
   has an implementation in the reference; Line/Previous are serialisation tags without
   semantics (-> HGI_ERR_UNSUPPORTED).  LeftTop (src/interpolator.rs:15-28) has no tag. */
typedef enum {
    HGI_INTERP_CROSSED = 0,
    HGI_INTERP_LINE = 1,
    HGI_INTERP_PREVIOUS = 2,
    HGI_INTERP_LEFTTOP = 3
} hgi_interp_t;

/* src/quantizator.rs:17 `NoOp`, :36 `Linear`. */
typedef enum { HGI_QUANT_NOOP = 0, HGI_QUANT_LINEAR = 1 } hgi_quant_kind_t;

/* src/quantizator.rs:3-8 `QuantizationLevel` (values = bincode variant indices). */
typedef enum {
    HGI_QLEVEL_LOSSLESS = 0,
    HGI_QLEVEL_LOW = 1,
    HGI_QLEVEL_MEDIUM = 2,
    HGI_QLEVEL_HIGH = 3
} hgi_quant_level_t;

/* Which CUDA path a context uses.  All produce identical bytes. */
typedef enum {
    HGI_PATH_TILE = 0,         /* default: fused multi-level tile kernels (register-prefetch SWAR kernel where eligible) */
    HGI_PATH_PER_LEVEL = 1,    /* one kernel per level over HBM (north_star's literal shape) */
    HGI_PATH_TILE_GENERIC = 2, /* fused tiles, always the generic (scalar, any alignment) kernel */
    HGI_PATH_TILE_TMA = 3      /* fused tiles, persistent TMA-pipelined SWAR kernel instead of the prefetch one */
} hgi_path_t;

#define HGI_MAX_LEVELS 31u
/* Rows (width, pitch) must be shorter than this many bytes: the kernels keep tile-relative offsets in 32 bits. */
#define HGI_MAX_ROW_BYTES (1u << 26)

/* Encoder/decoder options: `Encoder::new(interpolator, quantizator, scale_level)`
   (src/encoder.rs:18-24) and `Decoder::new(interpolator)` + `levels` (src/decoder.rs:14-18). */
typedef struct {
    uint32_t levels;     /* scale_level; 0 => grid == image */
    int32_t interp;      /* hgi_interp_t */
    int32_t quant_kind;  /* hgi_quant_kind_t   (ignored by decode) */
    int32_t quant_level; /* hgi_quant_level_t  (ignored by decode and by NoOp) */
} hgi_params_t;

/* ---- library / context ------------------------------------------------------------------ */
int hgi_abi_version(void);
const char *hgi_strerror(int status);

/* Binds a context to CUDA device `device` (must be sm_100).  Holds the stream, scratch planes
   and staging buffers, so steady-state calls do not allocate. */
int hgi_ctx_create(int device, hgi_ctx_t **ctx_out);
void hgi_ctx_destroy(hgi_ctx_t *ctx);
int hgi_ctx_set_path(hgi_ctx_t *ctx, int path /* hgi_path_t */);
/* Host-pointer entry points stream a batch through `slots` (1..4) stream slots in chunks of `chunk_mb` MiB (H2D,
   kernels and D2H of different chunks overlap).  0 = the default (64 MiB, 3 slots; HGI_B200_CHUNK_MB and
   HGI_B200_SLOTS in the environment override the default).  A non-zero `chunk_mb` is also the chunk of
   hgi_histogram_u8 / hgi_error_metrics_u8 (MiB) and hgi_rgb_to_luma_u8 (Mi pixels), which alternate their chunks
   between two slots (defaults: 1024 / 256 MiB / 64 Mi pixels). */
int hgi_ctx_set_pipeline(hgi_ctx_t *ctx, uint32_t chunk_mb, uint32_t slots);
int hgi_ctx_synchronize(hgi_ctx_t *ctx);
/* cudaError_t of the last failing runtime call (0 if none) and its string. */
int hgi_ctx_last_cuda_error(const hgi_ctx_t *ctx);
const char *hgi_ctx_last_cuda_error_string(const hgi_ctx_t *ctx);
/* Number of kernels this context has launched since creation (monotonic; kernels replayed from a captured
   launch chain count too), and how many of its device-API calls were served by one graph launch: identical
   consecutive `*_dev` calls whose chain has three or more kernels (levels > 4) are captured once and replayed
   (HGI_B200_GRAPHS=0 in the environment turns this off). */
uint64_t hgi_ctx_kernel_launches(const hgi_ctx_t *ctx);
uint64_t hgi_ctx_graph_launches(const hgi_ctx_t *ctx);

/* ---- page-locked host memory -------------------------------------------------------------- */
/* The host-pointer entry points copy with cudaMemcpyAsync: from/to pageable memory the driver stages every byte
   through its own buffers (a 1080p call then costs ~0.45 ms, almost all of it the two staged 2 MB copies); from/to
   page-locked memory the copy is one DMA (~0.1 ms per call).  hgi_host_alloc returns page-locked memory usable from
   every device (NULL on failure); hgi_host_register pins a buffer the caller already owns -- an image / grid buffer
   that is reused across calls -- until hgi_host_unregister.  Neither needs a context. */
void *hgi_host_alloc(size_t bytes);
void hgi_host_free(void *ptr);
int hgi_host_register(void *ptr, size_t bytes);
int hgi_host_unregister(void *ptr);

/* ---- quantizator ------------------------------------------------------------------------ */
/* `Linear::from(level)` / `NoOp::from(level)` (src/quantizator.rs:19-23,41-63): fills the
   256-entry table `quantize(v) = table[v]` and `error()` (:71-73).  Pure host arithmetic. */
int hgi_quant_table(int quant_kind, int quant_level, uint8_t table_out[256], uint8_t *error_out);

/* ---- host-pointer entry points (reference-facing) -------------------------------------- */
/* `Encoder::encode(&mut self, input: GrayImage) -> Grid` (src/encoder.rs:39-71).  `image` is not
   modified (the reference consumes it by value and clobbers it, :64); `grid_out` receives
   width*height residual bytes.  `recon_out` (nullable) receives the closed-loop reconstruction,
   i.e. the final state of the reference's `input` == what Decoder::decode will return. */
int hgi_encode_u8(hgi_ctx_t *ctx, const uint8_t *image, uint32_t width, uint32_t height,
                  const hgi_params_t *params, uint8_t *grid_out, uint8_t *recon_out);

/* `Decoder::decode(&mut self, (width,height), levels, &Grid) -> GrayImage`
   (src/decoder.rs:18-46). */
int hgi_decode_u8(hgi_ctx_t *ctx, const uint8_t *grid, uint32_t width, uint32_t height,
                  const hgi_params_t *params, uint8_t *image_out);

/* The same over `n_images` equally sized planes (one launch chain for the whole batch; copies
   are chunked and overlapped with the kernels).  `hist_out` (nullable) receives one 256-bin
   histogram of the residual bytes per image. */
int hgi_encode_batch_u8(hgi_ctx_t *ctx, const uint8_t *images, uint32_t n_images, uint32_t width,
                        uint32_t height, const hgi_params_t *params, uint8_t *grids_out,
                        uint32_t *hist_out /* [n_images][256] or NULL */);
int hgi_decode_batch_u8(hgi_ctx_t *ctx, const uint8_t *grids, uint32_t n_images, uint32_t width,
                        uint32_t height, const hgi_params_t *params, uint8_t *images_out);

/* Residual histogram / frequency table of `n` grid bytes (north_star's archive.rs stage; the
   reference leaves this to flate2 behind src/archive.rs:36-38).  hist_out[v] = #{bytes == v}. */
int hgi_histogram_u8(hgi_ctx_t *ctx, const uint8_t *grid, size_t n, uint64_t hist_out[256]);

/* `hgi test` error metrics (src/main.rs:84-92,106): sum of squared differences, its integer
   quotient by n (`sd /= uncompressed`), and the maximum absolute difference. */
int hgi_error_metrics_u8(hgi_ctx_t *ctx, const uint8_t *before, const uint8_t *after, size_t n,
                         uint64_t *sum_sq_out, uint64_t *sd_int_out, uint32_t *max_abs_out);

/* RGB8 (interleaved r,g,b) -> luma, the `to_luma()` of the `image` 0.19 crate that src/main.rs:42,74
   applies before encoding: l = 0.2126f*r + 0.7152f*g + 0.0722f*b in f32, left to right, every
   multiply and add rounded separately (no FMA), truncated to u8. */
int hgi_rgb_to_luma_u8(hgi_ctx_t *ctx, const uint8_t *rgb, size_t n_pixels, uint8_t *luma_out);

/* ---- device-pointer entry points (the timed ones) -------------------------------------- */
int hgi_encode_dev(hgi_ctx_t *ctx, const uint8_t *d_images, uint32_t n_images, uint32_t width,
                   uint32_t height, const hgi_params_t *params, uint8_t *d_grids_out,
                   uint8_t *d_recon_out /* nullable */,
                   uint32_t *d_hist_out /* nullable; [n_images][256], overwritten */,
                   void *stream);
int hgi_decode_dev(hgi_ctx_t *ctx, const uint8_t *d_grids, uint32_t n_images, uint32_t width,
                   uint32_t height, const hgi_params_t *params, uint8_t *d_images_out,
                   void *stream);
int hgi_rgb_to_luma_dev(hgi_ctx_t *ctx, const uint8_t *d_rgb, size_t n_pixels, uint8_t *d_luma_out,
                        void *stream);
int hgi_histogram_dev(hgi_ctx_t *ctx, const uint8_t *d_grid, size_t n_per_image,
                      uint32_t n_images, uint32_t *d_hist_out /* [n_images][256], overwritten */,
                      void *stream);
/* The same for planes whose rows are `pitch` bytes apart (pitch >= width; image k starts at k * pitch * height in
   every plane argument, all planes share the pitch).  A pitch that is a multiple of 16 with 16-byte-aligned bases
   puts any width on the 128-bit path: pad the rows of odd-width planes instead of packing them.  Input bytes in
   the padding are ignored; output bytes in the padding are unspecified.  pitch == width is hgi_encode_dev /
   hgi_decode_dev.  Not available on HGI_PATH_PER_LEVEL (-> HGI_ERR_UNSUPPORTED). */
int hgi_encode_dev_pitched(hgi_ctx_t *ctx, const uint8_t *d_images, uint32_t n_images, uint32_t width,
                           uint32_t height, uint32_t pitch, const hgi_params_t *params,
                           uint8_t *d_grids_out, uint8_t *d_recon_out /* nullable */,
                           uint32_t *d_hist_out /* nullable */, void *stream);
int hgi_decode_dev_pitched(hgi_ctx_t *ctx, const uint8_t *d_grids, uint32_t n_images, uint32_t width,
                           uint32_t height, uint32_t pitch, const hgi_params_t *params,
                           uint8_t *d_images_out, void *stream);
/* d_out[0] = sum of squares, d_out[1] = max abs (both u64, overwritten). */
int hgi_error_metrics_dev(hgi_ctx_t *ctx, const uint8_t *d_before, const uint8_t *d_after,
                          size_t n, uint64_t *d_out, void *stream);

/* ---- scalable decode: reduced resolution and region of interest ---------------------------- */
/* The grid is a pyramid: for scale_log2 = k the *scaled image* is ws x hs = ceil(width / 2^k) x ceil(height / 2^k)
   with scaled[v][u] = decode(grid)[v * 2^k][u * 2^k], and it equals the decode of the grid decimated by 2^k with
   L' = max(levels - k, 0) levels.  A region is a rectangle of the scaled image (scaled coordinates, inside it; NULL =
   the whole scaled image).  Because every dependency stays inside a coarse cell and its right / down neighbour, the
   region is decoded from a window of the decimated grid (DESIGN.md "Scalable decode"), byte-identical to slicing
   Decoder::decode (src/decoder.rs:18-46). */
typedef struct {
    uint32_t x, y, width, height;
} hgi_rect_t;
typedef struct {
    uint32_t scaled_width, scaled_height; /* ws, hs */
    uint32_t levels;                      /* L' = max(levels - scale_log2, 0): levels decoded on the window */
    hgi_rect_t window;                    /* decoded window of the scaled image (scaled coordinates) */
    uint32_t crop_x, crop_y;              /* the region's origin inside the window */
} hgi_region_plan_t;
/* The window of `region`: x0 = floor(u0 / A) * A with S' = 2^L', A = max(S', 16); x1 = min(ws, floor((u1 - 1) / S') * S'
   + 2 S' + 1); rows the same with A = S'.  Pure host arithmetic, no device needed.  HGI_ERR_INVALID_ARG: levels or
   scale_log2 > HGI_MAX_LEVELS, an empty region or one outside the scaled image, a NULL plan_out. */
int hgi_plan_region(uint32_t width, uint32_t height, uint32_t levels, uint32_t scale_log2, const hgi_rect_t *region,
                    hgi_region_plan_t *plan_out);
/* `n_images` grid planes (rows `pitch` bytes apart, as hgi_decode_dev_pitched) -> the region of each one's scaled
   image: d_out rows are `out_pitch` bytes apart (>= region width), planes out_pitch * region height apart, and no byte
   outside the rectangles is written.  Enqueued on `stream` like every *_dev call.  Not on HGI_PATH_PER_LEVEL
   (-> HGI_ERR_UNSUPPORTED). */
int hgi_decode_region_dev(hgi_ctx_t *ctx, const uint8_t *d_grids, uint32_t n_images, uint32_t width, uint32_t height,
                          uint32_t pitch, const hgi_params_t *params, uint32_t scale_log2, const hgi_rect_t *region,
                          uint8_t *d_out, uint32_t out_pitch, void *stream);
/* One host plane: only the window's grid rows (every 2^k-th row, the window's column span) go to the device and only
   the region (packed, region width x height bytes) comes back. */
int hgi_decode_region_u8(hgi_ctx_t *ctx, const uint8_t *grid, uint32_t width, uint32_t height,
                         const hgi_params_t *params, uint32_t scale_log2, const hgi_rect_t *region,
                         uint8_t *image_out);

/* ---- pool: the GPUs of one box behind one handle ------------------------------------------ */
/* The reference encodes one image per call on one thread (benches/bench.rs:54-110, src/main.rs:41-71); the path
   shards with no exchange between the shards (SURVEY.md 8e), so a pool drives one context per GPU from the calling
   thread: work is enqueued on every device before anything is waited for.  Results are byte-identical to a single
   context.  For overlap of the copies pass pinned (page-locked) host buffers. */
typedef struct hgi_pool hgi_pool_t;
/* `devices` = CUDA device ordinals (a device may appear more than once: several contexts on it);
   n_devices == 0 => every sm_100 device of the box. */
int hgi_pool_create(const int *devices, int n_devices, hgi_pool_t **pool_out);
void hgi_pool_destroy(hgi_pool_t *pool);
int hgi_pool_size(const hgi_pool_t *pool);
hgi_ctx_t *hgi_pool_ctx(hgi_pool_t *pool, int index);   /* the pool keeps ownership */
int hgi_pool_device(const hgi_pool_t *pool, int index); /* CUDA ordinal of member `index` */
int hgi_pool_synchronize(hgi_pool_t *pool);
/* By image: member k encodes/decodes the k-th contiguous share of the batch (`Encoder::encode` / `Decoder::decode`
   over n_images planes, src/encoder.rs:39-71, src/decoder.rs:18-46).  Host pointers; returns when all results are
   in the output buffers. */
int hgi_pool_encode_batch_u8(hgi_pool_t *pool, const uint8_t *images, uint32_t n_images, uint32_t width,
                             uint32_t height, const hgi_params_t *params, uint8_t *grids_out,
                             uint32_t *hist_out /* [n_images][256] or NULL */);
int hgi_pool_decode_batch_u8(hgi_pool_t *pool, const uint8_t *grids, uint32_t n_images, uint32_t width,
                             uint32_t height, const hgi_params_t *params, uint8_t *images_out);
/* By row band: ONE plane cut into at most hgi_pool_size() bands whose heights are multiples of S = 2^levels.
   Band [y0, y1) is computed by its member from the input rows [y0, in_y1), in_y1 = min(height, y1 + S + 1):
   the prediction of a cell reads only its own corners at floor and floor + step (src/interpolator.rs:67-73), so
   dependencies point right/down and the rows below a band are recomputed instead of exchanged. */
typedef struct {
    uint32_t y0, y1; /* output rows [y0, y1) */
    uint32_t in_y1;  /* input rows [y0, in_y1) */
} hgi_band_t;
int hgi_pool_plan_bands(const hgi_pool_t *pool, uint32_t height, uint32_t levels,
                        hgi_band_t *bands_out /* [hgi_pool_size()] */, int *n_bands_out);
/* The same plan for any number of bands (pure host arithmetic, no device needed): what a caller that runs one
   process per GPU uses to find the rows of its rank. */
int hgi_plan_bands(uint32_t height, uint32_t levels, uint32_t n_bands, hgi_band_t *bands_out /* [n_bands] */,
                   int *n_bands_out);
int hgi_pool_encode_plane_u8(hgi_pool_t *pool, const uint8_t *image, uint32_t width, uint32_t height,
                             const hgi_params_t *params, uint8_t *grid_out);
int hgi_pool_decode_plane_u8(hgi_pool_t *pool, const uint8_t *grid, uint32_t width, uint32_t height,
                             const hgi_params_t *params, uint8_t *image_out);
/* The same with the bands resident on their devices: d_bands_in[k] / d_bands_out[k] are buffers on the device of
   member k holding (in_y1 - y0) rows of `width` bytes of band k (input: the band and its overlap rows; output: rows
   [0, y1 - y0) are the result, the overlap rows are scratch).  Enqueues on every member's own stream and returns;
   hgi_pool_synchronize() waits.  Repeated calls with the same buffers replay one captured graph per device. */
int hgi_pool_encode_bands_dev(hgi_pool_t *pool, const uint8_t *const *d_bands_in, uint32_t width,
                              uint32_t height, const hgi_params_t *params, uint8_t *const *d_bands_out);
int hgi_pool_decode_bands_dev(hgi_pool_t *pool, const uint8_t *const *d_bands_in, uint32_t width,
                              uint32_t height, const hgi_params_t *params, uint8_t *const *d_bands_out);

/* ---- archive container (src/archive.rs) -------------------------------------------------- */
/* `Metadata` (src/archive.rs:15-22). */
typedef struct {
    uint32_t quantization_level; /* hgi_quant_level_t */
    uint32_t interpolation;      /* hgi_interp_t tag (Crossed/Line/Previous) */
    uint32_t width;
    uint32_t height;
    uint64_t scale_level;
} hgi_metadata_t;

#define HGI_ARCHIVE_MAGIC 0xBAADA555u /* src/archive.rs:13 */
#define HGI_ARCHIVE_HEADER_BYTES 28u  /* magic + bincode(Metadata) */

/* Upper bound of the serialised size for a grid of `n` bytes. */
size_t hgi_archive_bound(size_t n);
/* `Archive::serialize_to_writer` (src/archive.rs:31-41): MAGIC, bincode(metadata), then raw
   DEFLATE (best compression) of bincode(Grid{buffer, width}).  `grid_width` is Grid::width
   (src/grid.rs:4).  On success *out_len = bytes written. */
int hgi_archive_serialize(const hgi_metadata_t *metadata, const uint8_t *grid, size_t grid_len,
                          uint64_t grid_width, uint8_t *out, size_t out_capacity, size_t *out_len);
/* The same container with the entropy stage north_star describes: the residual frequency tables come from
   the GPU (hgi_histogram_* or the `hist_out` of encode) and the host only bit-packs.  `hist` holds `n_blocks`
   256-bin tables; table b describes grid bytes [b*block_bytes, min(grid_len, (b+1)*block_bytes)) (n_blocks == 1:
   the whole grid) and each block becomes one dynamic-Huffman DEFLATE block (literals only, no LZ77).  The
   result is a raw DEFLATE stream any inflate reads, i.e. `Archive::deserialize_from_reader` accepts it. */
size_t hgi_archive_huffman_bound(size_t n, size_t n_blocks);
int hgi_archive_serialize_huffman(const hgi_metadata_t *metadata, const uint8_t *grid, size_t grid_len,
                                  uint64_t grid_width, const uint32_t *hist, size_t n_blocks, size_t block_bytes,
                                  uint8_t *out, size_t out_capacity, size_t *out_len);
/* The entropy stage that is both small and fast: DEFLATE literals plus distance-1 matches ("repeat the previous
   byte"), one dynamic-Huffman block per table.  On residual planes of photographs the result is within a few per
   cent of zlib level 9 (no string matching is needed: a residual plane is runs of one symbol) at ~1/100 of its time.
   The 286-symbol literal/length frequency tables come from the GPU (hgi_rle_histogram_*): the parse is fixed --
   512-byte segments from the block start; per maximal run: one literal, matches of min(258, rest) while rest >= 3,
   the remaining 0..2 bytes as literals -- so the host only bit-packs.  `hist` holds `n_blocks` rows of
   HGI_RLE_TABLE_SYMBOLS counters; block_bytes must be a multiple of HGI_RLE_SEGMENT_BYTES when n_blocks > 1.
   A table that does not belong to the data is detected (HGI_ERR_INVALID_ARG). */
#define HGI_RLE_SEGMENT_BYTES 512u
#define HGI_RLE_TABLE_SYMBOLS 288u
int hgi_rle_histogram_u8(hgi_ctx_t *ctx, const uint8_t *grid, size_t n, size_t block_bytes, size_t n_blocks,
                         uint32_t *hist_out /* [n_blocks][HGI_RLE_TABLE_SYMBOLS] */);
int hgi_rle_histogram_dev(hgi_ctx_t *ctx, const uint8_t *d_grid, size_t n, size_t block_bytes, size_t n_blocks,
                          uint32_t *d_hist_out, void *stream);
int hgi_archive_serialize_rle(const hgi_metadata_t *metadata, const uint8_t *grid, size_t grid_len,
                              uint64_t grid_width, const uint32_t *hist, size_t n_blocks, size_t block_bytes,
                              uint8_t *out, size_t out_capacity, size_t *out_len);
/* `Archive::deserialize_from_reader` (src/archive.rs:43-55), split so the caller can allocate:
   _header parses MAGIC + metadata (28 bytes); _grid inflates the payload into `grid_out`. */
int hgi_archive_read_header(const uint8_t *data, size_t len, hgi_metadata_t *metadata_out);
int hgi_archive_read_grid(const uint8_t *data, size_t len, uint8_t *grid_out, size_t grid_capacity,
                          size_t *grid_len_out, uint64_t *grid_width_out);

#ifdef __cplusplus
}
#endif
#endif /* HGI_H_ */
