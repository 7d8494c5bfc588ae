"""Host-side mirror of the `hgi` crate's public surface (src/lib.rs:16-23) over the C ABI.

Names, argument meaning and error behaviour follow the reference:
  Encoder::new(interpolator, quantizator, scale_level) / encode(image) -> Grid   src/encoder.rs:18-71
  Decoder::new(interpolator) / decode((width,height), levels, &grid) -> image   src/decoder.rs:14-46
  Linear::from(QuantizationLevel) / NoOp::from(_), quantize(), error()          src/quantizator.rs:12-74
  Crossed / LeftTop, InterpolationType                                          src/interpolator.rs:4-30
  Archive{metadata, grid}.serialize_to_writer / deserialize_from_reader         src/archive.rs:24-55
All compute happens in libhgi_b200.so on the GPU; numpy arrays are only containers here.
"""
import collections
import ctypes
import enum
import threading

import numpy as np

from . import _lib
from ._lib import HgiError, Params, MetadataStruct, RectStruct, RegionPlanStruct


class QuantizationLevel(enum.IntEnum):      # src/quantizator.rs:3-8
    Lossless = 0
    Low = 1
    Medium = 2
    High = 3

    @classmethod
    def parse(cls, text):
        """clap `arg_enum!` parsing: case-insensitive variant names (src/options.rs:58-63)."""
        for v in cls:
            if v.name.lower() == str(text).lower():
                return v
        raise ValueError(f"valid values: {', '.join(v.name for v in cls)}")


class InterpolationType(enum.IntEnum):      # src/interpolator.rs:4-9 (serialisation tags)
    Crossed = 0
    Line = 1
    Previous = 2


_INTERP_LEFTTOP = 3
_QUANT_NOOP, _QUANT_LINEAR = 0, 1
PATH_TILE, PATH_PER_LEVEL, PATH_TILE_GENERIC, PATH_TILE_TMA = 0, 1, 2, 3


class Crossed:                              # src/interpolator.rs:30
    _id = int(InterpolationType.Crossed)


class LeftTop:                              # src/interpolator.rs:15
    _id = _INTERP_LEFTTOP


def _interp_id(interpolator):
    if isinstance(interpolator, type):
        interpolator = interpolator()
    if not hasattr(interpolator, "_id"):
        raise TypeError("interpolator must be Crossed or LeftTop")
    return interpolator._id


class _Quantizator:
    _kind = _QUANT_NOOP

    def __init__(self, level=QuantizationLevel.Lossless):
        self.level = QuantizationLevel(level)
        table = np.empty(256, np.uint8)
        err = ctypes.c_uint8(0)
        rc = _lib.lib().hgi_quant_table(self._kind, int(self.level), table.ctypes.data, ctypes.addressof(err))
        if rc:
            raise HgiError(rc, "hgi_quant_table")
        self.table, self._error = table, err.value

    @classmethod
    def from_level(cls, level):             # `From<QuantizationLevel>` (src/quantizator.rs:12)
        return cls(level)

    def quantize(self, value):              # src/quantizator.rs:13
        return int(self.table[int(value) & 0xFF])

    def error(self):                        # src/quantizator.rs:14
        return self._error


class NoOp(_Quantizator):                   # src/quantizator.rs:17-34
    _kind = _QUANT_NOOP


class Linear(_Quantizator):                 # src/quantizator.rs:36-74
    _kind = _QUANT_LINEAR


class Context:
    """One per GPU (hgi_ctx_t).  A process-wide default per device is created on first use."""
    _defaults = {}
    _lock = threading.Lock()

    def __init__(self, device=0, path=PATH_TILE):
        h = ctypes.c_void_p()
        rc = _lib.lib().hgi_ctx_create(int(device), ctypes.byref(h))
        if rc:
            raise HgiError(rc, "hgi_ctx_create")
        self._h = h
        self.device = int(device)
        if path != PATH_TILE:
            self.set_path(path)

    def set_path(self, path):
        rc = _lib.lib().hgi_ctx_set_path(self._h, int(path))
        if rc:
            raise HgiError(rc, "hgi_ctx_set_path")

    def set_pipeline(self, chunk_mb=0, slots=0):
        """Chunk size (MiB) and stream slots of the host-pointer entry points; 0 = default (hgi_ctx_set_pipeline)."""
        self.check(_lib.lib().hgi_ctx_set_pipeline(self._h, int(chunk_mb), int(slots)), "hgi_ctx_set_pipeline")

    def check(self, rc, where):
        if rc:
            raise HgiError(rc, where, _lib.lib().hgi_ctx_last_cuda_error_string(self._h).decode()
                           if rc == -3 else "")

    def synchronize(self):
        self.check(_lib.lib().hgi_ctx_synchronize(self._h), "hgi_ctx_synchronize")

    @property
    def kernel_launches(self):
        return int(_lib.lib().hgi_ctx_kernel_launches(self._h))

    @property
    def graph_launches(self):
        return int(_lib.lib().hgi_ctx_graph_launches(self._h))

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().hgi_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @classmethod
    def default(cls, device=0):
        with cls._lock:
            if device not in cls._defaults:
                cls._defaults[device] = cls(device)
            return cls._defaults[device]


class Pool:
    """hgi_pool_t: the GPUs of one box behind one handle (SURVEY.md 8e).  `devices` = CUDA ordinals (None: every
    sm_100 device); a device may be listed more than once."""

    def __init__(self, devices=None):
        h = ctypes.c_void_p()
        if devices is None:
            rc = _lib.lib().hgi_pool_create(None, 0, ctypes.byref(h))
        else:
            arr = (ctypes.c_int * len(devices))(*[int(d) for d in devices])
            rc = _lib.lib().hgi_pool_create(ctypes.cast(arr, ctypes.c_void_p), len(devices), ctypes.byref(h))
        if rc:
            raise HgiError(rc, "hgi_pool_create")
        self._h = h

    def __len__(self):
        return int(_lib.lib().hgi_pool_size(self._h))

    @property
    def devices(self):
        return [int(_lib.lib().hgi_pool_device(self._h, i)) for i in range(len(self))]

    def _check(self, rc, where):
        if rc:
            raise HgiError(rc, where)

    def synchronize(self):
        self._check(_lib.lib().hgi_pool_synchronize(self._h), "hgi_pool_synchronize")

    def plan_bands(self, height, levels):
        bands = (_lib.BandStruct * max(1, len(self)))()
        n = ctypes.c_int(0)
        self._check(_lib.lib().hgi_pool_plan_bands(self._h, int(height), int(levels), ctypes.cast(bands, ctypes.c_void_p),
                                                   ctypes.byref(n)), "hgi_pool_plan_bands")
        return [(bands[i].y0, bands[i].y1, bands[i].in_y1) for i in range(n.value)]

    def encode_batch(self, encoder, images, want_hist=False):
        imgs = _host_planes(images, "images")
        n, h, w = imgs.shape
        grids = np.empty_like(imgs)
        hist = np.zeros((n, 256), np.uint32) if want_hist else None
        p = encoder._p()
        self._check(_lib.lib().hgi_pool_encode_batch_u8(self._h, imgs.ctypes.data, n, w, h, ctypes.byref(p), grids.ctypes.data,
                                                        hist.ctypes.data if want_hist else None), "hgi_pool_encode_batch_u8")
        return (grids, hist) if want_hist else grids

    def decode_batch(self, decoder, levels, grids):
        g = _host_planes(grids, "grids")
        n, h, w = g.shape
        out = np.empty_like(g)
        p = _params(levels, decoder._interp)
        self._check(_lib.lib().hgi_pool_decode_batch_u8(self._h, g.ctypes.data, n, w, h, ctypes.byref(p), out.ctypes.data),
                    "hgi_pool_decode_batch_u8")
        return out

    def encode_plane(self, encoder, image):
        img = _host_planes(image, "image")
        h, w = img.shape
        grid = np.empty_like(img)
        p = encoder._p()
        self._check(_lib.lib().hgi_pool_encode_plane_u8(self._h, img.ctypes.data, w, h, ctypes.byref(p), grid.ctypes.data),
                    "hgi_pool_encode_plane_u8")
        return Grid(grid, w)

    def decode_plane(self, decoder, dimensions, levels, grid):
        width, height = int(dimensions[0]), int(dimensions[1])
        buf = grid.buffer if isinstance(grid, Grid) else _host_planes(grid, "grid").reshape(-1)
        out = np.empty((height, width), np.uint8)
        p = _params(levels, decoder._interp)
        self._check(_lib.lib().hgi_pool_decode_plane_u8(self._h, buf.ctypes.data, width, height, ctypes.byref(p), out.ctypes.data),
                    "hgi_pool_decode_plane_u8")
        return out

    def _band_ptrs(self, tensors):
        return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])

    def encode_bands_device(self, encoder, bands_in, width, height, bands_out):
        """bands_in[k] / bands_out[k]: CUDA uint8 tensors on the device of member k, (in_y1 - y0, width) each."""
        p = encoder._p()
        self._check(_lib.lib().hgi_pool_encode_bands_dev(self._h, ctypes.cast(self._band_ptrs(bands_in), ctypes.c_void_p), int(width), int(height),
                                                         ctypes.byref(p), ctypes.cast(self._band_ptrs(bands_out), ctypes.c_void_p)),
                    "hgi_pool_encode_bands_dev")

    def decode_bands_device(self, decoder, levels, bands_in, width, height, bands_out):
        p = _params(levels, decoder._interp)
        self._check(_lib.lib().hgi_pool_decode_bands_dev(self._h, ctypes.cast(self._band_ptrs(bands_in), ctypes.c_void_p), int(width), int(height),
                                                         ctypes.byref(p), ctypes.cast(self._band_ptrs(bands_out), ctypes.c_void_p)),
                    "hgi_pool_decode_bands_dev")

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().hgi_pool_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _params(levels, interp_id, quant=None):
    return Params(int(levels), int(interp_id), quant._kind if quant else 0, int(quant.level) if quant else 0)


def _host_planes(a, what):
    a = np.asarray(a)
    if a.dtype != np.uint8:
        raise TypeError(f"{what} must be uint8")
    if a.ndim not in (2, 3):
        raise ValueError(f"{what} must be (h, w) or (n, h, w)")
    return np.ascontiguousarray(a)


def _stream_handle(stream, device):
    """cudaStream_t for the C ABI.  The ABI reads NULL as "the context's own stream", so torch's
    legacy default stream (handle 0) is passed as cudaStreamLegacy (0x1)."""
    import torch
    h = stream if stream is not None else torch.cuda.current_stream(device).cuda_stream
    return h if h else 1


def _dev_planes(t, what):
    """(tensor as (n, h, w), n, h, w, pitch) for a CUDA uint8 tensor (n, h, w) or (h, w) whose rows are contiguous:
    either packed, or a `[..., :w]` view of a buffer with padded rows (pitch = stride of the row dimension)."""
    import torch
    v = t if t.dim() == 3 else t.unsqueeze(0)
    if not (v.is_cuda and v.dtype == torch.uint8 and v.dim() == 3):
        raise TypeError(f"{what} must be a CUDA uint8 tensor (n, h, w) or (h, w)")
    n, h, w = v.shape
    if n * h * w == 0 or v.is_contiguous():
        return v, n, h, w, w
    pitch = v.stride(1)
    if v.stride(2) != 1 or pitch < w or (n > 1 and v.stride(0) != pitch * h):
        raise ValueError(f"{what}: rows must be contiguous and images pitch * height bytes apart")
    return v, n, h, w, pitch


def _ctx_for(explicit, tensor):
    """The context of a device call: the explicit one (which must live on the tensor's device) or the per-device default."""
    dev = tensor.device.index if tensor.device.index is not None else 0
    if explicit is None:
        return Context.default(dev)
    if explicit.device != dev:
        raise ValueError(f"context is bound to cuda:{explicit.device} but the tensor lives on cuda:{dev}")
    return explicit


class Grid:
    """src/grid.rs:1-5: `buffer` (row-major u8, stride = width) + `width`."""

    def __init__(self, buffer, width):
        self.buffer = np.ascontiguousarray(buffer, dtype=np.uint8).reshape(-1)
        self.width = int(width)

    def as_plane(self):
        return self.buffer.reshape(-1, self.width) if self.width else self.buffer.reshape(0, 0)

    def get(self, column, line):            # src/grid.rs:24-27
        return int(self.buffer[line * self.width + column])

    def __eq__(self, other):
        return isinstance(other, Grid) and self.width == other.width and \
            self.buffer.shape == other.buffer.shape and bool((self.buffer == other.buffer).all())


class Encoder:
    """`Encoder<I, Q>` (src/encoder.rs:7-24)."""

    def __init__(self, interpolator, quantizator, scale_level, ctx=None):
        self.interpolator, self.quantizator, self.scale_level = interpolator, quantizator, int(scale_level)
        self._interp = _interp_id(interpolator)
        if not isinstance(quantizator, _Quantizator):
            raise TypeError("quantizator must be Linear or NoOp")
        self._ctx = ctx

    @property
    def ctx(self):
        return self._ctx or Context.default()

    def _p(self):
        return _params(self.scale_level, self._interp, self.quantizator)

    def encode(self, image, want_recon=False):
        """`encode(&mut self, input: GrayImage) -> Grid` (src/encoder.rs:39-71); host planes."""
        img = _host_planes(image, "image")
        if img.ndim != 2:
            raise ValueError("encode takes one (h, w) plane; use encode_batch")
        h, w = img.shape
        grid = np.empty_like(img)
        recon = np.empty_like(img) if want_recon else None
        p = self._p()
        rc = _lib.lib().hgi_encode_u8(self.ctx._h, img.ctypes.data, w, h, ctypes.byref(p), grid.ctypes.data,
                                      recon.ctypes.data if want_recon else None)
        self.ctx.check(rc, "hgi_encode_u8")
        g = Grid(grid, w)
        return (g, recon) if want_recon else g

    def encode_batch(self, images, want_hist=False):
        imgs = _host_planes(images, "images")
        if imgs.ndim != 3:
            raise ValueError("encode_batch takes (n, h, w)")
        n, h, w = imgs.shape
        grids = np.empty_like(imgs)
        hist = np.zeros((n, 256), np.uint32) if want_hist else None
        p = self._p()
        rc = _lib.lib().hgi_encode_batch_u8(self.ctx._h, imgs.ctypes.data, n, w, h, ctypes.byref(p),
                                            grids.ctypes.data, hist.ctypes.data if want_hist else None)
        self.ctx.check(rc, "hgi_encode_batch_u8")
        return (grids, hist) if want_hist else grids

    def encode_device(self, images, grids_out=None, recon_out=None, hist_out=None, stream=None):
        """Device-resident batch: `images` is a CUDA uint8 torch tensor (n, h, w) or (h, w), packed or with padded
        rows (see _dev_planes); the outputs must have the same layout."""
        import torch
        t, n, h, w, pitch = _dev_planes(images, "images")
        ctx = _ctx_for(self._ctx, t)
        if grids_out is None:
            grids_out = torch.empty_strided(t.shape, t.stride(), dtype=torch.uint8, device=t.device)
        for o, what in ((grids_out, "grids_out"), (recon_out, "recon_out")):
            if o is not None and _dev_planes(o, what)[1:] != (n, h, w, pitch):
                raise ValueError(f"{what} must have the shape and row pitch of images")
        st = _stream_handle(stream, t.device)
        p = self._p()
        rc = _lib.lib().hgi_encode_dev_pitched(ctx._h, t.data_ptr(), n, w, h, pitch, ctypes.byref(p), grids_out.data_ptr(),
                                               recon_out.data_ptr() if recon_out is not None else None,
                                               hist_out.data_ptr() if hist_out is not None else None, st)
        ctx.check(rc, "hgi_encode_dev_pitched")
        return grids_out if grids_out.dim() == images.dim() else grids_out[0]


class Decoder:
    """`Decoder<I>` (src/decoder.rs:6-16)."""

    def __init__(self, interpolator, ctx=None):
        self.interpolator = interpolator
        self._interp = _interp_id(interpolator)
        self._ctx = ctx

    @property
    def ctx(self):
        return self._ctx or Context.default()

    def decode(self, dimensions, levels, grid):
        """`decode(&mut self, (width, height), levels, &Grid) -> GrayImage` (src/decoder.rs:18-46)."""
        width, height = int(dimensions[0]), int(dimensions[1])
        buf = grid.buffer if isinstance(grid, Grid) else _host_planes(grid, "grid").reshape(-1)
        if buf.size != width * height:
            raise ValueError("grid size does not match dimensions")
        out = np.empty((height, width), np.uint8)
        p = _params(levels, self._interp)
        rc = _lib.lib().hgi_decode_u8(self.ctx._h, buf.ctypes.data, width, height, ctypes.byref(p), out.ctypes.data)
        self.ctx.check(rc, "hgi_decode_u8")
        return out

    def decode_batch(self, levels, grids):
        g = _host_planes(grids, "grids")
        n, h, w = g.shape
        out = np.empty_like(g)
        p = _params(levels, self._interp)
        rc = _lib.lib().hgi_decode_batch_u8(self.ctx._h, g.ctypes.data, n, w, h, ctypes.byref(p), out.ctypes.data)
        self.ctx.check(rc, "hgi_decode_batch_u8")
        return out

    def decode_device(self, levels, grids, images_out=None, stream=None):
        import torch
        t, n, h, w, pitch = _dev_planes(grids, "grids")
        ctx = _ctx_for(self._ctx, t)
        if images_out is None:
            images_out = torch.empty_strided(t.shape, t.stride(), dtype=torch.uint8, device=t.device)
        if _dev_planes(images_out, "images_out")[1:] != (n, h, w, pitch):
            raise ValueError("images_out must have the shape and row pitch of grids")
        st = _stream_handle(stream, t.device)
        p = _params(levels, self._interp)
        rc = _lib.lib().hgi_decode_dev_pitched(ctx._h, t.data_ptr(), n, w, h, pitch, ctypes.byref(p), images_out.data_ptr(), st)
        ctx.check(rc, "hgi_decode_dev_pitched")
        return images_out if images_out.dim() == grids.dim() else images_out[0]

    def decode_region(self, dimensions, levels, grid, region=None, scale_log2=0):
        """Scalable decode of one host grid: `decode(dimensions, levels, grid)[::2^k, ::2^k]` cut to `region` =
        (x, y, width, height) in those scaled coordinates (None: the whole scaled image), byte for byte, computed from
        the window of grid rows the region depends on (hgi_decode_region_u8)."""
        width, height = int(dimensions[0]), int(dimensions[1])
        buf = grid.buffer if isinstance(grid, Grid) else _host_planes(grid, "grid").reshape(-1)
        if buf.size != width * height:
            raise ValueError("grid size does not match dimensions")
        rw, rh = _region_size(width, height, levels, scale_log2, region)
        out = np.empty((rh, rw), np.uint8)
        p = _params(levels, self._interp)
        rc = _lib.lib().hgi_decode_region_u8(self.ctx._h, buf.ctypes.data, width, height, ctypes.byref(p), int(scale_log2),
                                             _rect(region), out.ctypes.data)
        self.ctx.check(rc, "hgi_decode_region_u8")
        return out

    def decode_region_device(self, levels, grids, region=None, scale_log2=0, out=None, stream=None):
        """The same for CUDA grids (n, h, w) or (h, w), packed or with padded rows (hgi_decode_region_dev): the result
        is (n, rh, rw) (or (rh, rw)); `out` may be such a tensor with padded rows, whose padding is left untouched."""
        import torch
        t, n, h, w, pitch = _dev_planes(grids, "grids")
        ctx = _ctx_for(self._ctx, t)
        rw, rh = _region_size(w, h, levels, scale_log2, region)
        if out is None:
            out = torch.empty((n, rh, rw) if grids.dim() == 3 else (rh, rw), dtype=torch.uint8, device=t.device)
        o, on, oh, ow, out_pitch = _dev_planes(out, "out")
        if (on, oh, ow) != (n, rh, rw) or o.device != t.device:
            raise ValueError(f"out must be ({n}, {rh}, {rw}) on {t.device}")
        st = _stream_handle(stream, t.device)
        p = _params(levels, self._interp)
        rc = _lib.lib().hgi_decode_region_dev(ctx._h, t.data_ptr(), n, w, h, pitch, ctypes.byref(p), int(scale_log2),
                                              _rect(region), o.data_ptr(), out_pitch, st)
        ctx.check(rc, "hgi_decode_region_dev")
        return out


RegionPlan = collections.namedtuple("RegionPlan", "scaled_width scaled_height levels window crop_x crop_y")
RegionPlan.__doc__ = """hgi_region_plan_t: the scaled image's size, the levels decoded on the window (L' = max(L - k, 0)),
the window (x, y, width, height) in scaled coordinates and the region's origin inside it."""


def _rect(region):
    """hgi_rect_t* for an (x, y, width, height) region; None = the whole scaled image (NULL)."""
    if region is None:
        return None
    x, y, w, h = (int(v) for v in region)
    if min(x, y, w, h) < 0:
        raise ValueError("region must be (x, y, width, height) with non-negative values")
    return ctypes.byref(RectStruct(x, y, w, h))


def plan_region(width, height, levels, scale_log2=0, region=None):
    """hgi_plan_region: the window a scalable decode of `region` (scaled coordinates; None = the whole scaled image)
    reads.  Pure host arithmetic."""
    p = RegionPlanStruct()
    rc = _lib.lib().hgi_plan_region(int(width), int(height), int(levels), int(scale_log2), _rect(region), ctypes.byref(p))
    if rc:
        raise HgiError(rc, "hgi_plan_region")
    w = p.window
    return RegionPlan(p.scaled_width, p.scaled_height, p.levels, (w.x, w.y, w.width, w.height), p.crop_x, p.crop_y)


def _region_size(width, height, levels, scale_log2, region):
    if region is not None:
        return int(region[2]), int(region[3])
    pl = plan_region(width, height, levels, scale_log2)
    return pl.scaled_width, pl.scaled_height


def histogram(grid, ctx=None):
    """Residual frequency table: hist[v] = #{grid bytes == v} (north_star's archive.rs stage)."""
    ctx = ctx or Context.default()
    buf = grid.buffer if isinstance(grid, Grid) else np.ascontiguousarray(grid, dtype=np.uint8).reshape(-1)
    hist = np.zeros(256, np.uint64)
    ctx.check(_lib.lib().hgi_histogram_u8(ctx._h, buf.ctypes.data, buf.size, hist.ctypes.data), "hgi_histogram_u8")
    return hist


def error_metrics(before, after, ctx=None):
    """`hgi test` numbers (src/main.rs:84-111): dict(sum_sq, sd_int, max_abs, sd=sqrt(sd_int))."""
    ctx = ctx or Context.default()
    b = np.ascontiguousarray(before, dtype=np.uint8).reshape(-1)
    a = np.ascontiguousarray(after, dtype=np.uint8).reshape(-1)
    if a.size != b.size:
        raise ValueError("size mismatch")
    s, q, m = ctypes.c_uint64(0), ctypes.c_uint64(0), ctypes.c_uint32(0)
    rc = _lib.lib().hgi_error_metrics_u8(ctx._h, b.ctypes.data, a.ctypes.data, b.size, ctypes.addressof(s),
                                         ctypes.addressof(q), ctypes.addressof(m))
    ctx.check(rc, "hgi_error_metrics_u8")
    return {"sum_sq": s.value, "sd_int": q.value, "max_abs": m.value, "sd": float(q.value) ** 0.5}


def rgb_to_luma(rgb, ctx=None):
    """`image::DynamicImage::to_luma()` as called at src/main.rs:42,74 (f32 weights, no FMA, truncation).
    `rgb` is (h, w, 3) uint8; returns the (h, w) luma plane the codec consumes."""
    ctx = ctx or Context.default()
    a = np.ascontiguousarray(rgb, dtype=np.uint8)
    if a.ndim != 3 or a.shape[2] != 3:
        raise ValueError("rgb must be (h, w, 3)")
    out = np.empty(a.shape[:2], np.uint8)
    ctx.check(_lib.lib().hgi_rgb_to_luma_u8(ctx._h, a.ctypes.data, out.size, out.ctypes.data), "hgi_rgb_to_luma_u8")
    return out


class Metadata:
    """src/archive.rs:15-22."""

    def __init__(self, quantization_level, interpolation, width, height, scale_level):
        self.quantization_level = QuantizationLevel(quantization_level)
        self.interpolation = InterpolationType(interpolation)
        self.width, self.height, self.scale_level = int(width), int(height), int(scale_level)

    def _struct(self):
        return MetadataStruct(int(self.quantization_level), int(self.interpolation), self.width, self.height,
                              self.scale_level)

    def __eq__(self, other):
        return isinstance(other, Metadata) and vars(self) == vars(other)

    def __repr__(self):
        return f"Metadata({vars(self)})"


class Archive:
    """src/archive.rs:24-55."""
    MAGIC = 0xBAADA555

    def __init__(self, metadata, grid):
        self.metadata, self.grid = metadata, grid

    def __eq__(self, other):
        return isinstance(other, Archive) and self.metadata == other.metadata and self.grid == other.grid

    def serialize_to_writer(self, w, entropy="deflate", hist=None, block_rows=None, ctx=None):
        """entropy="deflate": zlib level-9 raw DEFLATE (the stand-in for flate2's Compression::best()).
        entropy="rle": literals + distance-1 matches, token tables from the GPU (hgi_rle_histogram_u8 unless `hist`
        carries the (n_blocks, 288) tables), host bit-packing (hgi_archive_serialize_rle): zlib-9 size on residual
        planes at ~1/100 of its time; blocks are `block_rows` rows rounded to 512-byte multiples.
        entropy="huffman": GPU-built frequency tables + host bit-packing (hgi_archive_serialize_huffman);
        `hist` may carry the (n_blocks, 256) tables already produced by encode, else they are computed on the
        GPU here, one table per `block_rows` grid rows (default: one table for the whole grid)."""
        L = _lib.lib()
        buf = self.grid.buffer
        n = ctypes.c_size_t(0)
        m = self.metadata._struct()
        if entropy == "deflate":
            cap = L.hgi_archive_bound(buf.size)
            out = np.empty(cap, np.uint8)
            rc = L.hgi_archive_serialize(ctypes.byref(m), buf.ctypes.data, buf.size, self.grid.width, out.ctypes.data,
                                         cap, ctypes.byref(n))
            if rc:
                raise HgiError(rc, "hgi_archive_serialize")
        elif entropy == "huffman":
            block = buf.size if not block_rows else int(block_rows) * self.grid.width
            block = max(1, min(block, max(buf.size, 1)))
            n_blocks = max(1, -(-buf.size // block))
            if hist is None:
                hist = np.stack([histogram(buf[b * block:(b + 1) * block], ctx=ctx) for b in range(n_blocks)])
            hist = np.ascontiguousarray(np.asarray(hist).reshape(n_blocks, 256), dtype=np.uint32)
            cap = L.hgi_archive_huffman_bound(buf.size, n_blocks)
            out = np.empty(cap, np.uint8)
            rc = L.hgi_archive_serialize_huffman(ctypes.byref(m), buf.ctypes.data, buf.size, self.grid.width,
                                                 hist.ctypes.data, n_blocks, block, out.ctypes.data, cap, ctypes.byref(n))
            if rc:
                raise HgiError(rc, "hgi_archive_serialize_huffman")
        elif entropy == "rle":
            seg = 512
            block = buf.size if not block_rows else -(-int(block_rows) * self.grid.width // seg) * seg
            block = max(1, min(block, max(buf.size, 1)))
            n_blocks = max(1, -(-buf.size // block))
            if hist is None:
                hist = np.zeros((n_blocks, 288), np.uint32)
                c = ctx or Context.default()
                c.check(L.hgi_rle_histogram_u8(c._h, buf.ctypes.data if buf.size else None, buf.size, block, n_blocks,
                                               hist.ctypes.data), "hgi_rle_histogram_u8")
            hist = np.ascontiguousarray(np.asarray(hist).reshape(n_blocks, 288), dtype=np.uint32)
            cap = L.hgi_archive_huffman_bound(buf.size, n_blocks)
            out = np.empty(cap, np.uint8)
            rc = L.hgi_archive_serialize_rle(ctypes.byref(m), buf.ctypes.data, buf.size, self.grid.width,
                                             hist.ctypes.data, n_blocks, block, out.ctypes.data, cap, ctypes.byref(n))
            if rc:
                raise HgiError(rc, "hgi_archive_serialize_rle")
        else:
            raise ValueError("entropy must be 'deflate', 'rle' or 'huffman'")
        w.write(out[:n.value].tobytes())

    @classmethod
    def deserialize_from_reader(cls, r):
        L = _lib.lib()
        data = np.frombuffer(r.read(), np.uint8)
        m = MetadataStruct()
        rc = L.hgi_archive_read_header(data.ctypes.data if data.size else None, data.size, ctypes.byref(m))
        if rc:
            raise HgiError(rc, "hgi_archive_read_header")
        glen, gw = ctypes.c_size_t(0), ctypes.c_uint64(0)
        # first call learns the length (bincode's u64 prefix), second call inflates into place
        rc = L.hgi_archive_read_grid(data.ctypes.data, data.size, None, 0, ctypes.byref(glen), ctypes.byref(gw))
        if rc not in (0, -7):
            raise HgiError(rc, "hgi_archive_read_grid")
        if glen.value > (1 << 40):
            raise HgiError(-6, "hgi_archive_read_grid", "implausible grid length")
        grid = np.empty(glen.value, np.uint8)
        rc = L.hgi_archive_read_grid(data.ctypes.data, data.size, grid.ctypes.data, grid.size, ctypes.byref(glen),
                                     ctypes.byref(gw))
        if rc:
            raise HgiError(rc, "hgi_archive_read_grid")
        md = Metadata(m.quantization_level, m.interpolation, m.width, m.height, m.scale_level)
        return cls(md, Grid(grid, gw.value))
