//! Raw bindings of `include/hgi.h` (libhgi_b200.so).  Source only: not compiled in the repository's build image.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct hgi_ctx_t {
    _private: [u8; 0],
}

#[repr(C)]
pub struct hgi_pool_t {
    _private: [u8; 0],
}

/// One row band of `hgi_pool_plan_bands`: output rows `[y0, y1)`, input rows `[y0, in_y1)`.
#[repr(C)]
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub struct hgi_band_t {
    pub y0: u32,
    pub y1: u32,
    pub in_y1: u32,
}

/// A rectangle of the scaled image of a scalable decode (scaled coordinates).
#[repr(C)]
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub struct hgi_rect_t {
    pub x: u32,
    pub y: u32,
    pub width: u32,
    pub height: u32,
}

/// `hgi_plan_region`: the scaled size, the levels decoded on the window, the window and the region's origin in it.
#[repr(C)]
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub struct hgi_region_plan_t {
    pub scaled_width: u32,
    pub scaled_height: u32,
    pub levels: u32,
    pub window: hgi_rect_t,
    pub crop_x: u32,
    pub crop_y: u32,
}

pub const HGI_ABI_VERSION: c_int = 2;
pub const HGI_OK: c_int = 0;
pub const HGI_ERR_INVALID_ARG: c_int = -1;
pub const HGI_ERR_NO_DEVICE: c_int = -2;
pub const HGI_ERR_CUDA: c_int = -3;
pub const HGI_ERR_ALLOC: c_int = -4;
pub const HGI_ERR_BAD_MAGIC: c_int = -5;
pub const HGI_ERR_TRUNCATED: c_int = -6;
pub const HGI_ERR_BUFFER_TOO_SMALL: c_int = -7;
pub const HGI_ERR_UNSUPPORTED: c_int = -8;

pub const HGI_INTERP_CROSSED: i32 = 0; // InterpolationType::Crossed (src/interpolator.rs:6)
pub const HGI_INTERP_LEFTTOP: i32 = 3; // LeftTop (src/interpolator.rs:15), no serialisation tag
pub const HGI_QUANT_NOOP: i32 = 0; // src/quantizator.rs:17
pub const HGI_QUANT_LINEAR: i32 = 1; // src/quantizator.rs:36

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct hgi_params_t {
    pub levels: u32,
    pub interp: i32,
    pub quant_kind: i32,
    pub quant_level: i32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub struct hgi_metadata_t {
    pub quantization_level: u32,
    pub interpolation: u32,
    pub width: u32,
    pub height: u32,
    pub scale_level: u64,
}

extern "C" {
    pub fn hgi_abi_version() -> c_int;
    pub fn hgi_strerror(status: c_int) -> *const c_char;
    pub fn hgi_ctx_create(device: c_int, ctx_out: *mut *mut hgi_ctx_t) -> c_int;
    pub fn hgi_ctx_destroy(ctx: *mut hgi_ctx_t);
    /// Accepts 0..=3 (hgi_path_t); every value runs the fused tile path, the others are kept for compatibility.
    pub fn hgi_ctx_set_path(ctx: *mut hgi_ctx_t, path: c_int) -> c_int;
    pub fn hgi_ctx_set_pipeline(ctx: *mut hgi_ctx_t, chunk_mb: u32, slots: u32) -> c_int;
    pub fn hgi_ctx_synchronize(ctx: *mut hgi_ctx_t) -> c_int;
    pub fn hgi_ctx_last_cuda_error(ctx: *const hgi_ctx_t) -> c_int;
    pub fn hgi_ctx_last_cuda_error_string(ctx: *const hgi_ctx_t) -> *const c_char;
    pub fn hgi_ctx_kernel_launches(ctx: *const hgi_ctx_t) -> u64;
    pub fn hgi_ctx_graph_launches(ctx: *const hgi_ctx_t) -> u64;
    pub fn hgi_host_alloc(bytes: usize) -> *mut c_void;
    pub fn hgi_host_free(ptr: *mut c_void);
    pub fn hgi_host_register(ptr: *mut c_void, bytes: usize) -> c_int;
    pub fn hgi_host_unregister(ptr: *mut c_void) -> c_int;
    pub fn hgi_quant_table(kind: c_int, level: c_int, table_out: *mut u8, error_out: *mut u8) -> c_int;
    pub fn hgi_encode_u8(ctx: *mut hgi_ctx_t, image: *const u8, width: u32, height: u32, params: *const hgi_params_t,
                         grid_out: *mut u8, recon_out: *mut u8) -> c_int;
    pub fn hgi_decode_u8(ctx: *mut hgi_ctx_t, grid: *const u8, width: u32, height: u32, params: *const hgi_params_t,
                         image_out: *mut u8) -> c_int;
    pub fn hgi_encode_batch_u8(ctx: *mut hgi_ctx_t, images: *const u8, n_images: u32, width: u32, height: u32,
                               params: *const hgi_params_t, grids_out: *mut u8, hist_out: *mut u32) -> c_int;
    pub fn hgi_decode_batch_u8(ctx: *mut hgi_ctx_t, grids: *const u8, n_images: u32, width: u32, height: u32,
                               params: *const hgi_params_t, images_out: *mut u8) -> c_int;
    pub fn hgi_histogram_u8(ctx: *mut hgi_ctx_t, grid: *const u8, n: usize, hist_out: *mut u64) -> c_int;
    pub fn hgi_error_metrics_u8(ctx: *mut hgi_ctx_t, before: *const u8, after: *const u8, n: usize,
                                sum_sq_out: *mut u64, sd_int_out: *mut u64, max_abs_out: *mut u32) -> c_int;
    pub fn hgi_rgb_to_luma_u8(ctx: *mut hgi_ctx_t, rgb: *const u8, n_pixels: usize, luma_out: *mut u8) -> c_int;
    pub fn hgi_encode_dev(ctx: *mut hgi_ctx_t, d_images: *const u8, n_images: u32, width: u32, height: u32,
                          params: *const hgi_params_t, d_grids_out: *mut u8, d_recon_out: *mut u8,
                          d_hist_out: *mut u32, stream: *mut c_void) -> c_int;
    pub fn hgi_decode_dev(ctx: *mut hgi_ctx_t, d_grids: *const u8, n_images: u32, width: u32, height: u32,
                          params: *const hgi_params_t, d_images_out: *mut u8, stream: *mut c_void) -> c_int;
    pub fn hgi_encode_dev_pitched(ctx: *mut hgi_ctx_t, d_images: *const u8, n_images: u32, width: u32, height: u32,
                                  pitch: u32, params: *const hgi_params_t, d_grids_out: *mut u8, d_recon_out: *mut u8,
                                  d_hist_out: *mut u32, stream: *mut c_void) -> c_int;
    pub fn hgi_decode_dev_pitched(ctx: *mut hgi_ctx_t, d_grids: *const u8, n_images: u32, width: u32, height: u32,
                                  pitch: u32, params: *const hgi_params_t, d_images_out: *mut u8,
                                  stream: *mut c_void) -> c_int;
    pub fn hgi_rgb_to_luma_dev(ctx: *mut hgi_ctx_t, d_rgb: *const u8, n_pixels: usize, d_luma_out: *mut u8,
                               stream: *mut c_void) -> c_int;
    pub fn hgi_histogram_dev(ctx: *mut hgi_ctx_t, d_grid: *const u8, n_per_image: usize, n_images: u32,
                             d_hist_out: *mut u32, stream: *mut c_void) -> c_int;
    pub fn hgi_error_metrics_dev(ctx: *mut hgi_ctx_t, d_before: *const u8, d_after: *const u8, n: usize,
                                 d_out: *mut u64, stream: *mut c_void) -> c_int;
    pub fn hgi_plan_region(width: u32, height: u32, levels: u32, scale_log2: u32, region: *const hgi_rect_t,
                           plan_out: *mut hgi_region_plan_t) -> c_int;
    pub fn hgi_decode_region_dev(ctx: *mut hgi_ctx_t, d_grids: *const u8, n_images: u32, width: u32, height: u32,
                                 pitch: u32, params: *const hgi_params_t, scale_log2: u32, region: *const hgi_rect_t,
                                 d_out: *mut u8, out_pitch: u32, stream: *mut c_void) -> c_int;
    pub fn hgi_decode_region_u8(ctx: *mut hgi_ctx_t, grid: *const u8, width: u32, height: u32,
                                params: *const hgi_params_t, scale_log2: u32, region: *const hgi_rect_t,
                                image_out: *mut u8) -> c_int;
    pub fn hgi_plan_crop(width: u32, height: u32, levels: u32, scale_log2: u32, crop: *const hgi_rect_t,
                         plan_out: *mut hgi_region_plan_t) -> c_int;
    pub fn hgi_decode_crops_dev(ctx: *mut hgi_ctx_t, d_grids: *const u8, n_images: u32, width: u32, height: u32,
                                pitch: u32, params: *const hgi_params_t, scale_log2: u32, crop_width: u32,
                                crop_height: u32, d_origins: *const i32, d_out: *mut u8, out_pitch: u32,
                                stream: *mut c_void) -> c_int;
    pub fn hgi_pool_create(devices: *const c_int, n_devices: c_int, pool_out: *mut *mut hgi_pool_t) -> c_int;
    pub fn hgi_pool_destroy(pool: *mut hgi_pool_t);
    pub fn hgi_pool_size(pool: *const hgi_pool_t) -> c_int;
    pub fn hgi_pool_ctx(pool: *mut hgi_pool_t, index: c_int) -> *mut hgi_ctx_t;
    pub fn hgi_pool_device(pool: *const hgi_pool_t, index: c_int) -> c_int;
    pub fn hgi_pool_synchronize(pool: *mut hgi_pool_t) -> c_int;
    pub fn hgi_pool_encode_batch_u8(pool: *mut hgi_pool_t, images: *const u8, n_images: u32, width: u32, height: u32,
                                    params: *const hgi_params_t, grids_out: *mut u8, hist_out: *mut u32) -> c_int;
    pub fn hgi_pool_decode_batch_u8(pool: *mut hgi_pool_t, grids: *const u8, n_images: u32, width: u32, height: u32,
                                    params: *const hgi_params_t, images_out: *mut u8) -> c_int;
    pub fn hgi_plan_bands(height: u32, levels: u32, n_bands: u32, bands_out: *mut hgi_band_t, n_bands_out: *mut c_int) -> c_int;
    pub fn hgi_pool_plan_bands(pool: *const hgi_pool_t, height: u32, levels: u32, bands_out: *mut hgi_band_t,
                               n_bands_out: *mut c_int) -> c_int;
    pub fn hgi_pool_encode_plane_u8(pool: *mut hgi_pool_t, image: *const u8, width: u32, height: u32,
                                    params: *const hgi_params_t, grid_out: *mut u8) -> c_int;
    pub fn hgi_pool_decode_plane_u8(pool: *mut hgi_pool_t, grid: *const u8, width: u32, height: u32,
                                    params: *const hgi_params_t, image_out: *mut u8) -> c_int;
    pub fn hgi_pool_encode_bands_dev(pool: *mut hgi_pool_t, d_bands_in: *const *const u8, width: u32, height: u32,
                                     params: *const hgi_params_t, d_bands_out: *const *mut u8) -> c_int;
    pub fn hgi_pool_decode_bands_dev(pool: *mut hgi_pool_t, d_bands_in: *const *const u8, width: u32, height: u32,
                                     params: *const hgi_params_t, d_bands_out: *const *mut u8) -> c_int;
    pub fn hgi_archive_bound(n: usize) -> usize;
    pub fn hgi_archive_serialize(m: *const hgi_metadata_t, grid: *const u8, grid_len: usize, grid_width: u64,
                                 out: *mut u8, out_capacity: usize, out_len: *mut usize) -> c_int;
    pub fn hgi_archive_huffman_bound(n: usize, n_blocks: usize) -> usize;
    pub fn hgi_archive_serialize_huffman(m: *const hgi_metadata_t, grid: *const u8, grid_len: usize, grid_width: u64,
                                         hist: *const u32, n_blocks: usize, block_bytes: usize, out: *mut u8,
                                         out_capacity: usize, out_len: *mut usize) -> c_int;
    pub fn hgi_rle_histogram_u8(ctx: *mut hgi_ctx_t, grid: *const u8, n: usize, block_bytes: usize, n_blocks: usize,
                                hist_out: *mut u32) -> c_int;
    pub fn hgi_rle_histogram_dev(ctx: *mut hgi_ctx_t, d_grid: *const u8, n: usize, block_bytes: usize, n_blocks: usize,
                                 d_hist_out: *mut u32, stream: *mut c_void) -> c_int;
    pub fn hgi_archive_serialize_rle(m: *const hgi_metadata_t, grid: *const u8, grid_len: usize, grid_width: u64,
                                     hist: *const u32, n_blocks: usize, block_bytes: usize, out: *mut u8,
                                     out_capacity: usize, out_len: *mut usize) -> c_int;
    pub fn hgi_archive_read_header(data: *const u8, len: usize, m: *mut hgi_metadata_t) -> c_int;
    pub fn hgi_archive_read_grid(data: *const u8, len: usize, grid_out: *mut u8, grid_capacity: usize,
                                 grid_len_out: *mut usize, grid_width_out: *mut u64) -> c_int;
}
