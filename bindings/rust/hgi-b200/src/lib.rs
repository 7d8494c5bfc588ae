//! Safe wrappers over `hgi-sys` with the names and signatures of the reference crate `hgi`
//! (src/lib.rs:16-23): drop-in replacements for `Encoder` / `Decoder` and their option types.
//! Source only: not compiled in the repository's build image (no Rust toolchain there).
extern crate hgi_sys;
extern crate image;

use hgi_sys::*;
use image::GrayImage;
use std::ffi::CStr;
use std::ptr;
use std::sync::Once;

/// src/quantizator.rs:3-8
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum QuantizationLevel { Lossless = 0, Low = 1, Medium = 2, High = 3 }

/// src/interpolator.rs:4-9 (serialisation tags)
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum InterpolationType { Crossed = 0, Line = 1, Previous = 2 }

/// src/interpolator.rs:11-13 -- the arithmetic lives in the CUDA kernels; the trait only selects the variant.
pub trait Interpolator { const ID: i32; }
pub struct Crossed;  // src/interpolator.rs:30
pub struct LeftTop;  // src/interpolator.rs:15
impl Interpolator for Crossed { const ID: i32 = HGI_INTERP_CROSSED; }
impl Interpolator for LeftTop { const ID: i32 = HGI_INTERP_LEFTTOP; }

/// src/quantizator.rs:12-15
pub trait Quantizator: From<QuantizationLevel> {
    const KIND: i32;
    fn level(&self) -> QuantizationLevel;
    fn quantize(&self, value: u8) -> u8;
    fn error(&self) -> u8;
}

fn table_of(kind: i32, level: QuantizationLevel) -> ([u8; 256], u8) {
    let mut table = [0u8; 256];
    let mut error = 0u8;
    let rc = unsafe { hgi_quant_table(kind, level as i32, table.as_mut_ptr(), &mut error) };
    assert_eq!(rc, HGI_OK);
    (table, error)
}

/// src/quantizator.rs:17-34
pub struct NoOp;
impl From<QuantizationLevel> for NoOp { fn from(_: QuantizationLevel) -> Self { NoOp } }
impl Quantizator for NoOp {
    const KIND: i32 = HGI_QUANT_NOOP;
    fn level(&self) -> QuantizationLevel { QuantizationLevel::Lossless }
    fn quantize(&self, value: u8) -> u8 { value }
    fn error(&self) -> u8 { 0 }
}

/// src/quantizator.rs:36-74
pub struct Linear { table: [u8; 256], error: u8, level: QuantizationLevel }
impl From<QuantizationLevel> for Linear {
    fn from(level: QuantizationLevel) -> Self {
        let (table, error) = table_of(HGI_QUANT_LINEAR, level);
        Linear { table, error, level }
    }
}
impl Quantizator for Linear {
    const KIND: i32 = HGI_QUANT_LINEAR;
    fn level(&self) -> QuantizationLevel { self.level }
    fn quantize(&self, value: u8) -> u8 { self.table[value as usize] }
    fn error(&self) -> u8 { self.error }
}

/// src/grid.rs:1-5
#[derive(Debug, PartialEq, Eq)]
pub struct Grid { pub buffer: Vec<u8>, pub width: usize }
impl Grid {
    pub unsafe fn get(&self, column: u32, line: u32) -> u8 { *self.buffer.get_unchecked(line as usize * self.width + column as usize) }
}

struct Ctx(*mut hgi_ctx_t);
unsafe impl Sync for Ctx {}
static mut CTX: Ctx = Ctx(ptr::null_mut());
static INIT: Once = Once::new();

/// One process-wide context on device 0 (HGI_B200_DEVICE overrides).  Calls on one context must not be issued
/// from several threads at once; create one `hgi_ctx_t` per thread / GPU with `hgi_sys` directly for that.
fn ctx() -> *mut hgi_ctx_t {
    unsafe {
        INIT.call_once(|| {
            let dev = std::env::var("HGI_B200_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
            let mut c = ptr::null_mut();
            let rc = hgi_ctx_create(dev, &mut c);
            assert_eq!(rc, HGI_OK, "hgi_ctx_create: {}", strerror(rc));
            CTX = Ctx(c);
        });
        CTX.0
    }
}

fn strerror(rc: i32) -> String { unsafe { CStr::from_ptr(hgi_strerror(rc)).to_string_lossy().into_owned() } }

/// src/encoder.rs:7-24
pub struct Encoder<I, Q> { _interpolator: I, quantizator: Q, scale_level: usize }

impl<I: Interpolator, Q: Quantizator> Encoder<I, Q> {
    pub fn new(interpolator: I, quantizator: Q, scale_level: usize) -> Self {
        Encoder { _interpolator: interpolator, quantizator, scale_level }
    }

    /// src/encoder.rs:39-71 -- `input` is consumed like in the reference; the GPU never modifies it.
    pub fn encode(&mut self, input: GrayImage) -> Grid {
        let (width, height) = input.dimensions();
        let mut buffer = vec![0u8; width as usize * height as usize];
        let params = hgi_params_t { levels: self.scale_level as u32, interp: I::ID, quant_kind: Q::KIND,
                                    quant_level: self.quantizator.level() as i32 };
        let rc = unsafe { hgi_encode_u8(ctx(), input.as_ptr(), width, height, &params, buffer.as_mut_ptr(), ptr::null_mut()) };
        assert_eq!(rc, HGI_OK, "hgi_encode_u8: {}", strerror(rc));   // encode is infallible in the reference
        Grid { buffer, width: width as usize }
    }
}

/// src/decoder.rs:6-16
pub struct Decoder<I> { _interpolator: I }

impl<I: Interpolator> Decoder<I> {
    pub fn new(interpolator: I) -> Self { Decoder { _interpolator: interpolator } }

    /// src/decoder.rs:18-46
    pub fn decode(&mut self, (width, height): (u32, u32), levels: usize, grid: &Grid) -> GrayImage {
        let mut image = GrayImage::new(width, height);
        assert_eq!(grid.buffer.len(), width as usize * height as usize);
        let params = hgi_params_t { levels: levels as u32, interp: I::ID, quant_kind: HGI_QUANT_NOOP, quant_level: 0 };
        let rc = unsafe { hgi_decode_u8(ctx(), grid.buffer.as_ptr(), width, height, &params, image.as_mut_ptr()) };
        assert_eq!(rc, HGI_OK, "hgi_decode_u8: {}", strerror(rc));
        image
    }

    /// Scalable decode (not in the reference): `decode(..)` at 1/2^scale_log2 resolution -- every 2^k-th pixel of
    /// every 2^k-th row -- cut to `region` (x, y, width, height in those scaled coordinates; None = all of it).
    /// Only the grid rows the region depends on are decoded.  An empty or out-of-image region is an error.
    pub fn decode_region(&mut self, (width, height): (u32, u32), levels: usize, grid: &Grid, scale_log2: u32,
                         region: Option<(u32, u32, u32, u32)>) -> Result<GrayImage, String> {
        if grid.buffer.len() != width as usize * height as usize {
            return Err("grid size does not match dimensions".into());
        }
        let plan = plan_region(width, height, levels as u32, scale_log2, region)?;
        let (rw, rh) = region.map_or((plan.scaled_width, plan.scaled_height), |r| (r.2, r.3));
        let rect = region.map(|(x, y, w, h)| hgi_rect_t { x, y, width: w, height: h });
        let mut image = GrayImage::new(rw, rh);
        let params = hgi_params_t { levels: levels as u32, interp: I::ID, quant_kind: HGI_QUANT_NOOP, quant_level: 0 };
        let rc = unsafe {
            hgi_decode_region_u8(ctx(), grid.buffer.as_ptr(), width, height, &params, scale_log2,
                                 rect.as_ref().map_or(ptr::null(), |r| r as *const hgi_rect_t), image.as_mut_ptr())
        };
        if rc != HGI_OK { return Err(format!("hgi_decode_region_u8: {}", strerror(rc))); }
        Ok(image)
    }
}

/// `hgi_plan_region`: the window of the grid a scalable decode of `region` reads (pure host arithmetic).
pub fn plan_region(width: u32, height: u32, levels: u32, scale_log2: u32, region: Option<(u32, u32, u32, u32)>)
                   -> Result<hgi_region_plan_t, String> {
    let rect = region.map(|(x, y, w, h)| hgi_rect_t { x, y, width: w, height: h });
    let mut plan = hgi_region_plan_t { scaled_width: 0, scaled_height: 0, levels: 0,
                                       window: hgi_rect_t { x: 0, y: 0, width: 0, height: 0 }, crop_x: 0, crop_y: 0 };
    let rc = unsafe {
        hgi_plan_region(width, height, levels, scale_log2, rect.as_ref().map_or(ptr::null(), |r| r as *const hgi_rect_t),
                        &mut plan)
    };
    if rc != HGI_OK { return Err(format!("hgi_plan_region: {}", strerror(rc))); }
    Ok(plan)
}

/// `hgi_plan_crop`: the window every plane of a batched crop of this size decodes, placed for the origin `crop.0, crop.1`
/// (pure host arithmetic).  Its width and height depend on the crop's size only.
pub fn plan_crop(width: u32, height: u32, levels: u32, scale_log2: u32, crop: (u32, u32, u32, u32))
                 -> Result<hgi_region_plan_t, String> {
    let rect = hgi_rect_t { x: crop.0, y: crop.1, width: crop.2, height: crop.3 };
    let mut plan = hgi_region_plan_t { scaled_width: 0, scaled_height: 0, levels: 0,
                                       window: hgi_rect_t { x: 0, y: 0, width: 0, height: 0 }, crop_x: 0, crop_y: 0 };
    let rc = unsafe { hgi_plan_crop(width, height, levels, scale_log2, &rect, &mut plan) };
    if rc != HGI_OK { return Err(format!("hgi_plan_crop: {}", strerror(rc))); }
    Ok(plan)
}
