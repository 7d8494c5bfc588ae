"""ctypes binding of libhgi_b200.so (include/hgi.h).  Loading is strict: if the library is not
built, importing fails loudly -- there is no Python or CPU implementation to fall back to."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HGI_B200_LIB") or os.path.join(_HERE, "libhgi_b200.so")


class HgiLibraryError(RuntimeError):
    pass


class HgiError(RuntimeError):
    def __init__(self, status, where, detail=""):
        self.status = status
        msg = lib().hgi_strerror(status).decode()
        super().__init__(f"{where}: {msg} (status {status}){(' - ' + detail) if detail else ''}")


class Params(ctypes.Structure):
    _fields_ = [("levels", ctypes.c_uint32), ("interp", ctypes.c_int32),
                ("quant_kind", ctypes.c_int32), ("quant_level", ctypes.c_int32)]


class BandStruct(ctypes.Structure):
    _fields_ = [("y0", ctypes.c_uint32), ("y1", ctypes.c_uint32), ("in_y1", ctypes.c_uint32)]


class RectStruct(ctypes.Structure):
    _fields_ = [("x", ctypes.c_uint32), ("y", ctypes.c_uint32), ("width", ctypes.c_uint32), ("height", ctypes.c_uint32)]


class RegionPlanStruct(ctypes.Structure):
    _fields_ = [("scaled_width", ctypes.c_uint32), ("scaled_height", ctypes.c_uint32), ("levels", ctypes.c_uint32),
                ("window", RectStruct), ("crop_x", ctypes.c_uint32), ("crop_y", ctypes.c_uint32)]


class MetadataStruct(ctypes.Structure):
    _fields_ = [("quantization_level", ctypes.c_uint32), ("interpolation", ctypes.c_uint32),
                ("width", ctypes.c_uint32), ("height", ctypes.c_uint32),
                ("scale_level", ctypes.c_uint64)]


_vp, _u32, _u64, _sz, _int = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_size_t, ctypes.c_int
_pp = ctypes.POINTER(Params)
_pm = ctypes.POINTER(MetadataStruct)
_pr = ctypes.POINTER(RectStruct)

# name -> (restype, argtypes); every function declared in include/hgi.h
PROTOTYPES = {
    "hgi_abi_version": (_int, []),
    "hgi_strerror": (ctypes.c_char_p, [_int]),
    "hgi_ctx_create": (_int, [_int, ctypes.POINTER(_vp)]),
    "hgi_ctx_destroy": (None, [_vp]),
    "hgi_ctx_set_path": (_int, [_vp, _int]),
    "hgi_ctx_set_pipeline": (_int, [_vp, _u32, _u32]),
    "hgi_ctx_synchronize": (_int, [_vp]),
    "hgi_ctx_last_cuda_error": (_int, [_vp]),
    "hgi_ctx_last_cuda_error_string": (ctypes.c_char_p, [_vp]),
    "hgi_ctx_kernel_launches": (_u64, [_vp]),
    "hgi_ctx_graph_launches": (_u64, [_vp]),
    "hgi_host_alloc": (_vp, [_sz]),
    "hgi_host_free": (None, [_vp]),
    "hgi_host_register": (_int, [_vp, _sz]),
    "hgi_host_unregister": (_int, [_vp]),
    "hgi_quant_table": (_int, [_int, _int, _vp, _vp]),
    "hgi_encode_u8": (_int, [_vp, _vp, _u32, _u32, _pp, _vp, _vp]),
    "hgi_decode_u8": (_int, [_vp, _vp, _u32, _u32, _pp, _vp]),
    "hgi_encode_batch_u8": (_int, [_vp, _vp, _u32, _u32, _u32, _pp, _vp, _vp]),
    "hgi_decode_batch_u8": (_int, [_vp, _vp, _u32, _u32, _u32, _pp, _vp]),
    "hgi_histogram_u8": (_int, [_vp, _vp, _sz, _vp]),
    "hgi_error_metrics_u8": (_int, [_vp, _vp, _vp, _sz, _vp, _vp, _vp]),
    "hgi_rgb_to_luma_u8": (_int, [_vp, _vp, _sz, _vp]),
    "hgi_rgb_to_luma_dev": (_int, [_vp, _vp, _sz, _vp, _vp]),
    "hgi_encode_dev": (_int, [_vp, _vp, _u32, _u32, _u32, _pp, _vp, _vp, _vp, _vp]),
    "hgi_decode_dev": (_int, [_vp, _vp, _u32, _u32, _u32, _pp, _vp, _vp]),
    "hgi_encode_dev_pitched": (_int, [_vp, _vp, _u32, _u32, _u32, _u32, _pp, _vp, _vp, _vp, _vp]),
    "hgi_decode_dev_pitched": (_int, [_vp, _vp, _u32, _u32, _u32, _u32, _pp, _vp, _vp]),
    "hgi_histogram_dev": (_int, [_vp, _vp, _sz, _u32, _vp, _vp]),
    "hgi_error_metrics_dev": (_int, [_vp, _vp, _vp, _sz, _vp, _vp]),
    "hgi_plan_region": (_int, [_u32, _u32, _u32, _u32, _pr, ctypes.POINTER(RegionPlanStruct)]),
    "hgi_decode_region_dev": (_int, [_vp, _vp, _u32, _u32, _u32, _u32, _pp, _u32, _pr, _vp, _u32, _vp]),
    "hgi_decode_region_u8": (_int, [_vp, _vp, _u32, _u32, _pp, _u32, _pr, _vp]),
    "hgi_pool_create": (_int, [_vp, _int, ctypes.POINTER(_vp)]),
    "hgi_pool_destroy": (None, [_vp]),
    "hgi_pool_size": (_int, [_vp]),
    "hgi_pool_ctx": (_vp, [_vp, _int]),
    "hgi_pool_device": (_int, [_vp, _int]),
    "hgi_pool_synchronize": (_int, [_vp]),
    "hgi_pool_encode_batch_u8": (_int, [_vp, _vp, _u32, _u32, _u32, _pp, _vp, _vp]),
    "hgi_pool_decode_batch_u8": (_int, [_vp, _vp, _u32, _u32, _u32, _pp, _vp]),
    "hgi_plan_bands": (_int, [_u32, _u32, _u32, _vp, ctypes.POINTER(_int)]),
    "hgi_pool_plan_bands": (_int, [_vp, _u32, _u32, _vp, ctypes.POINTER(_int)]),
    "hgi_pool_encode_plane_u8": (_int, [_vp, _vp, _u32, _u32, _pp, _vp]),
    "hgi_pool_decode_plane_u8": (_int, [_vp, _vp, _u32, _u32, _pp, _vp]),
    "hgi_pool_encode_bands_dev": (_int, [_vp, _vp, _u32, _u32, _pp, _vp]),
    "hgi_pool_decode_bands_dev": (_int, [_vp, _vp, _u32, _u32, _pp, _vp]),
    "hgi_archive_bound": (_sz, [_sz]),
    "hgi_archive_serialize": (_int, [_pm, _vp, _sz, _u64, _vp, _sz, ctypes.POINTER(_sz)]),
    "hgi_archive_huffman_bound": (_sz, [_sz, _sz]),
    "hgi_archive_serialize_huffman": (_int, [_pm, _vp, _sz, _u64, _vp, _sz, _sz, _vp, _sz, ctypes.POINTER(_sz)]),
    "hgi_rle_histogram_u8": (_int, [_vp, _vp, _sz, _sz, _sz, _vp]),
    "hgi_rle_histogram_dev": (_int, [_vp, _vp, _sz, _sz, _sz, _vp, _vp]),
    "hgi_archive_serialize_rle": (_int, [_pm, _vp, _sz, _u64, _vp, _sz, _sz, _vp, _sz, ctypes.POINTER(_sz)]),
    "hgi_archive_read_header": (_int, [_vp, _sz, _pm]),
    "hgi_archive_read_grid": (_int, [_vp, _sz, _vp, _sz, ctypes.POINTER(_sz), ctypes.POINTER(_u64)]),
}

ABI_VERSION = 2      # HGI_ABI_VERSION of include/hgi.h

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HgiLibraryError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C rustyhgi_b200/csrc`.  rustyhgi_b200 has no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError => ABI mismatch, fail loudly
            fn.restype = res
            fn.argtypes = args
        if L.hgi_abi_version() != ABI_VERSION:
            raise HgiLibraryError(f"ABI version {L.hgi_abi_version()} != {ABI_VERSION}")
        _lib = L
    return _lib
