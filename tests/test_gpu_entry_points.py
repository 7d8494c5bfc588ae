"""Status codes and kernel counts of every entry point of include/hgi.h that takes a context or a pool (-m gpu).

The status table pins the order of the argument checks: handle, parameters, plane size, an empty job (OK, whatever its
pointers), data pointers -- and the checks only some entry points make (u32 histogram bins, out_pitch, the region plan,
RLE blocks, pipeline and path ranges).  The launch table pins hgi_ctx_kernel_launches after one small valid call of each
entry point: a pool charges each member for its own kernels, a replayed launch chain counts its kernels, and a call that
only clears its output (a zero-length histogram) counts none.  Every buffer is a few KB."""
import ctypes

import numpy as np
import pytest

import rustyhgi_b200 as hgi
from tile_model import expected_launches

pytestmark = pytest.mark.gpu

W, H, N = 64, 48, 2
INVALID, UNSUPPORTED = -1, -8
BIG = 1 << 26                          # HGI_MAX_ROW_BYTES


def prm(levels=4, interp=0, kind=1, qlevel=2):
    return ctypes.byref(hgi._lib.Params(levels, interp, kind, qlevel))


@pytest.fixture(scope="module")
def env():
    import torch
    L = hgi.lib()
    ctxs = {p: hgi.Context(0, p) for p in (hgi.PATH_TILE, hgi.PATH_PER_LEVEL, hgi.PATH_TILE_GENERIC)}
    pool = hgi.Pool([0, 0])
    rng = np.random.default_rng(7)
    host = rng.integers(0, 256, 1 << 16, dtype=np.uint8)
    hout = np.zeros(1 << 16, np.uint8)
    dev = torch.from_numpy(host).cuda()
    dout = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    dhist = torch.zeros(4 * 288, dtype=torch.int32, device="cuda")
    yield L, ctxs, pool, host, hout, dev, dout, dhist
    torch.cuda.synchronize()
    pool.close()
    for c in ctxs.values():
        c.close()


def entry_calls(L, host, hout, dev, dout):
    """name -> (call(handle, params, w, h, n, pitch, src, dst), handle, family).  `src` / `dst` of False: a null
    pointer; of True: a valid buffer of this call's memory kind."""
    hb, ho, db, do = host.ctypes.data, hout.ctypes.data, dev.data_ptr(), dout.data_ptr()
    hh = hout.ctypes.data + 32768      # u32 bins of the host-API histograms

    def H_(s, d):
        return (hb if s else None), (ho if d else None)

    def D_(s, d):
        return (db if s else None), (do if d else None)

    bands_in = (ctypes.c_void_p * 2)(db, db)
    bands_out = (ctypes.c_void_p * 2)(do, do + 8192)
    null_band = (ctypes.c_void_p * 2)(db, None)

    def bands(s, d):
        return (ctypes.cast(bands_in, ctypes.c_void_p) if s else None), (ctypes.cast(bands_out, ctypes.c_void_p) if d else None)

    c = {
        "hgi_encode_u8": (lambda h, p, w, ht, n, pi, s, d: L.hgi_encode_u8(h, H_(s, d)[0], w, ht, p, H_(s, d)[1], None), "ctx", "enc1"),
        "hgi_decode_u8": (lambda h, p, w, ht, n, pi, s, d: L.hgi_decode_u8(h, H_(s, d)[0], w, ht, p, H_(s, d)[1]), "ctx", "dec1"),
        "hgi_encode_batch_u8": (lambda h, p, w, ht, n, pi, s, d: L.hgi_encode_batch_u8(h, H_(s, d)[0], n, w, ht, p, H_(s, d)[1], hh), "ctx", "enc"),
        "hgi_decode_batch_u8": (lambda h, p, w, ht, n, pi, s, d: L.hgi_decode_batch_u8(h, H_(s, d)[0], n, w, ht, p, H_(s, d)[1]), "ctx", "dec"),
        "hgi_encode_dev": (lambda h, p, w, ht, n, pi, s, d: L.hgi_encode_dev(h, D_(s, d)[0], n, w, ht, p, D_(s, d)[1], None, None, None), "ctx", "enc"),
        "hgi_decode_dev": (lambda h, p, w, ht, n, pi, s, d: L.hgi_decode_dev(h, D_(s, d)[0], n, w, ht, p, D_(s, d)[1], None), "ctx", "dec"),
        "hgi_encode_dev_pitched": (lambda h, p, w, ht, n, pi, s, d: L.hgi_encode_dev_pitched(h, D_(s, d)[0], n, w, ht, pi, p, D_(s, d)[1], None, None, None), "ctx", "encp"),
        "hgi_decode_dev_pitched": (lambda h, p, w, ht, n, pi, s, d: L.hgi_decode_dev_pitched(h, D_(s, d)[0], n, w, ht, pi, p, D_(s, d)[1], None), "ctx", "decp"),
        "hgi_decode_region_dev": (lambda h, p, w, ht, n, pi, s, d: L.hgi_decode_region_dev(h, D_(s, d)[0], n, w, ht, pi, p, 1, None, D_(s, d)[1], 64, None), "ctx", "region"),
        "hgi_decode_region_u8": (lambda h, p, w, ht, n, pi, s, d: L.hgi_decode_region_u8(h, H_(s, d)[0], w, ht, p, 1, None, H_(s, d)[1]), "ctx", "region1"),
        "hgi_pool_encode_batch_u8": (lambda h, p, w, ht, n, pi, s, d: L.hgi_pool_encode_batch_u8(h, H_(s, d)[0], n, w, ht, p, H_(s, d)[1], None), "pool", "enc"),
        "hgi_pool_decode_batch_u8": (lambda h, p, w, ht, n, pi, s, d: L.hgi_pool_decode_batch_u8(h, H_(s, d)[0], n, w, ht, p, H_(s, d)[1]), "pool", "dec"),
        "hgi_pool_encode_plane_u8": (lambda h, p, w, ht, n, pi, s, d: L.hgi_pool_encode_plane_u8(h, H_(s, d)[0], w, ht, p, H_(s, d)[1]), "pool", "enc1"),
        "hgi_pool_decode_plane_u8": (lambda h, p, w, ht, n, pi, s, d: L.hgi_pool_decode_plane_u8(h, H_(s, d)[0], w, ht, p, H_(s, d)[1]), "pool", "dec1"),
        "hgi_pool_encode_bands_dev": (lambda h, p, w, ht, n, pi, s, d: L.hgi_pool_encode_bands_dev(h, bands(s, d)[0], w, ht, p, bands(s, d)[1]), "pool", "enc1"),
        "hgi_pool_decode_bands_dev": (lambda h, p, w, ht, n, pi, s, d: L.hgi_pool_decode_bands_dev(h, bands(s, d)[0], w, ht, p, bands(s, d)[1]), "pool", "dec1"),
    }
    return c, null_band


def test_status_codes(env):
    L, ctxs, pool, host, hout, dev, dout, dhist = env
    ctx = ctxs[hgi.PATH_TILE]._h
    calls, null_band = entry_calls(L, host, hout, dev, dout)
    got, want = {}, {}

    def case(tag, rc, expect):
        got[tag], want[tag] = rc, expect

    for name, (f, kind, fam) in calls.items():
        h = ctx if kind == "ctx" else pool._h
        enc, n = fam.startswith("enc"), (1 if fam.endswith("1") else N)
        pitched = fam in ("encp", "decp", "region")
        region = fam.startswith("region")
        bands_dev = name.endswith("_bands_dev")

        def run(p=None, w=W, ht=H, nn=n, pi=W, s=True, d=True, handle=h):
            return f(handle, p if p is not None else prm(), w, ht, nn, pi, s, d)

        case((name, "null handle"), run(handle=None), INVALID)
        case((name, "levels 32"), run(p=prm(levels=32)), INVALID)
        case((name, "interp Line"), run(p=prm(interp=1)), UNSUPPORTED)
        case((name, "interp Previous"), run(p=prm(interp=2)), UNSUPPORTED)
        case((name, "interp 9"), run(p=prm(interp=9)), INVALID)
        case((name, "quant_kind 5"), run(p=prm(kind=5)), INVALID if enc else 0)
        case((name, "quant_level 4"), run(p=prm(qlevel=4)), INVALID if enc else 0)
        case((name, "quant_level -1"), run(p=prm(qlevel=-1)), INVALID if enc else 0)
        case((name, "NoOp, any level"), run(p=prm(kind=0, qlevel=9)), 0)
        case((name, "row of 2^26 bytes"), run(w=BIG, ht=1, pi=BIG), INVALID)
        if pitched:
            case((name, "pitch < width"), run(pi=W - 1), INVALID)
            case((name, "pitch 2^26"), run(pi=BIG), INVALID)
        case((name, "null source"), run(s=False), INVALID)
        case((name, "null destination"), run(d=False), INVALID)
        # an empty job is OK whatever its data pointers; the band arrays are checked with the handle
        case((name, "empty plane, null pointers"), run(w=0, s=False, d=False), INVALID if (region or bands_dev) else 0)
        case((name, "empty plane, bad params first"), run(p=prm(interp=1), w=0, s=False, d=False),
             INVALID if bands_dev else UNSUPPORTED)
        if n > 1:
            case((name, "no images, null pointers"), run(nn=0, s=False, d=False), 0)
    # bands: a null member pointer
    for name in ("hgi_pool_encode_bands_dev", "hgi_pool_decode_bands_dev"):
        case((name, "null band"), getattr(L, name)(pool._h, ctypes.cast(null_band, ctypes.c_void_p), W, H, prm(),
                                                   ctypes.cast(null_band, ctypes.c_void_p)), INVALID)
    # checks only some entry points make
    hb, db, do, dh = host.ctypes.data, dev.data_ptr(), dout.data_ptr(), dhist.data_ptr()
    case("encode_dev: u32 bins, empty job", L.hgi_encode_dev(ctx, db, 0, 1 << 16, 1 << 16, prm(), do, None, dh, None), INVALID)
    case("encode_dev: u32 bins, bad interp", L.hgi_encode_dev(ctx, db, 0, 1 << 16, 1 << 16, prm(interp=1), do, None, dh, None), UNSUPPORTED)
    rect = ctypes.byref(hgi._lib.RectStruct(0, 0, 10, 10))
    case("region_dev: out_pitch < width", L.hgi_decode_region_dev(ctx, db, 1, W, H, W, prm(), 0, rect, do, 9, None), INVALID)
    case("region_dev: out_pitch before empty", L.hgi_decode_region_dev(ctx, None, 0, W, H, W, prm(), 0, rect, None, 9, None), INVALID)
    bad = ctypes.byref(hgi._lib.RectStruct(60, 0, 10, 10))
    case("region_dev: region outside, no images", L.hgi_decode_region_dev(ctx, None, 0, W, H, W, prm(), 0, bad, None, 64, None), INVALID)
    case("region_u8: region outside", L.hgi_decode_region_u8(ctx, hb, W, H, prm(), 0, bad, hb), INVALID)
    case("region_dev: scale 32", L.hgi_decode_region_dev(ctx, db, 1, W, H, W, prm(), 32, None, do, 64, None), INVALID)
    # every path value runs the tile path, which takes regions and padded rows
    pl = ctxs[hgi.PATH_PER_LEVEL]._h
    for k in (0, 1):
        case(("path 1 region", k), L.hgi_decode_region_dev(pl, db, 1, W, H, W, prm(), k, rect, do, 64, None), 0)
        case(("path 1 region u8", k), L.hgi_decode_region_u8(pl, hb, W, H, prm(), k, rect, hout.ctypes.data), 0)
    case("path 1 pitched encode", L.hgi_encode_dev_pitched(pl, db, 1, W, H, W + 16, prm(), do, None, None, None), 0)
    case("path 1 pitched decode", L.hgi_decode_dev_pitched(pl, db, 1, W, H, W + 16, prm(), do, None), 0)
    case("path 1 packed encode", L.hgi_encode_dev_pitched(pl, db, 1, W, H, W, prm(), do, None, None, None), 0)
    # histograms, reductions, colour conversion
    keep = [np.zeros(256, np.uint64), np.zeros(4 * 288, np.uint32)] + [np.zeros(1, np.uint64) for _ in range(3)]
    hist64, rle_out, *mp = [a.ctypes.data for a in keep]
    for tag, rc, expect in (
            ("histogram_dev: null handle", L.hgi_histogram_dev(None, db, 64, 1, dh, None), INVALID),
            ("histogram_dev: null hist", L.hgi_histogram_dev(ctx, db, 64, 1, None, None), INVALID),
            ("histogram_dev: 2^32 per image", L.hgi_histogram_dev(ctx, db, 1 << 32, 0, dh, None), INVALID),
            ("histogram_dev: no images, null grid", L.hgi_histogram_dev(ctx, None, 64, 0, dh, None), 0),
            ("histogram_dev: null grid", L.hgi_histogram_dev(ctx, None, 64, 1, dh, None), INVALID),
            ("histogram_dev: empty planes, null grid", L.hgi_histogram_dev(ctx, None, 0, 2, dh, None), 0),
            ("histogram_u8: null handle", L.hgi_histogram_u8(None, hb, 64, hist64), INVALID),
            ("histogram_u8: null hist", L.hgi_histogram_u8(ctx, hb, 64, None), INVALID),
            ("histogram_u8: empty, null grid", L.hgi_histogram_u8(ctx, None, 0, hist64), 0),
            ("histogram_u8: null grid", L.hgi_histogram_u8(ctx, None, 64, hist64), INVALID),
            ("error_metrics_dev: null handle", L.hgi_error_metrics_dev(None, db, db, 64, dh, None), INVALID),
            ("error_metrics_dev: null out", L.hgi_error_metrics_dev(ctx, db, db, 64, None, None), INVALID),
            ("error_metrics_dev: null input", L.hgi_error_metrics_dev(ctx, db, None, 64, dh, None), INVALID),
            ("error_metrics_dev: empty, null inputs", L.hgi_error_metrics_dev(ctx, None, None, 0, dh, None), 0),
            ("error_metrics_u8: null handle", L.hgi_error_metrics_u8(None, hb, hb, 64, *mp), INVALID),
            ("error_metrics_u8: null input", L.hgi_error_metrics_u8(ctx, None, hb, 64, *mp), INVALID),
            ("error_metrics_u8: empty, null everything", L.hgi_error_metrics_u8(ctx, None, None, 0, None, None, None), 0),
            ("rgb_to_luma_dev: null handle", L.hgi_rgb_to_luma_dev(None, db, 64, do, None), INVALID),
            ("rgb_to_luma_dev: empty, null pointers", L.hgi_rgb_to_luma_dev(ctx, None, 0, None, None), 0),
            ("rgb_to_luma_dev: null output", L.hgi_rgb_to_luma_dev(ctx, db, 64, None, None), INVALID),
            ("rgb_to_luma_dev: 2^60 + 1 pixels", L.hgi_rgb_to_luma_dev(ctx, db, (1 << 60) + 1, do, None), INVALID),
            ("rgb_to_luma_u8: null handle", L.hgi_rgb_to_luma_u8(None, hb, 64, hb), INVALID),
            ("rgb_to_luma_u8: empty, null pointers", L.hgi_rgb_to_luma_u8(ctx, None, 0, None), 0),
            ("rgb_to_luma_u8: null input", L.hgi_rgb_to_luma_u8(ctx, None, 64, hb), INVALID),
            ("rgb_to_luma_u8: 2^60 + 1 pixels", L.hgi_rgb_to_luma_u8(ctx, hb, (1 << 60) + 1, hb), INVALID),
            ("set_pipeline: null handle", L.hgi_ctx_set_pipeline(None, 0, 0), INVALID),
            ("set_pipeline: 4097 MiB", L.hgi_ctx_set_pipeline(ctx, 4097, 0), INVALID),
            ("set_pipeline: 5 slots", L.hgi_ctx_set_pipeline(ctx, 0, 5), INVALID),
            ("set_pipeline: 4096 MiB, 4 slots", L.hgi_ctx_set_pipeline(ctx, 4096, 4), 0),
            ("set_pipeline: defaults", L.hgi_ctx_set_pipeline(ctx, 0, 0), 0),
            ("set_path: null handle", L.hgi_ctx_set_path(None, 0), INVALID),
            ("set_path: -1", L.hgi_ctx_set_path(ctx, -1), INVALID),
            ("set_path: 4", L.hgi_ctx_set_path(ctx, 4), INVALID),
            ("set_path: 3", L.hgi_ctx_set_path(ctx, 3), 0),
            ("set_path: 0", L.hgi_ctx_set_path(ctx, 0), 0),
            ("synchronize: null handle", L.hgi_ctx_synchronize(None), INVALID),
            ("synchronize", L.hgi_ctx_synchronize(ctx), 0),
            ("pool_synchronize: null handle", L.hgi_pool_synchronize(None), INVALID),
            ("pool_synchronize", L.hgi_pool_synchronize(pool._h), 0),
            ("pool_plan_bands: null handle", L.hgi_pool_plan_bands(None, H, 4, rle_out, ctypes.byref(ctypes.c_int())), INVALID),
            ("pool_plan_bands: levels 32", L.hgi_pool_plan_bands(pool._h, H, 32, rle_out, ctypes.byref(ctypes.c_int())), INVALID)):
        case(tag, rc, expect)
    seg = 512    # HGI_RLE_SEGMENT_BYTES
    for name, f, dst in (("rle_histogram_dev", lambda *a: L.hgi_rle_histogram_dev(*a, None), dh),
                         ("rle_histogram_u8", L.hgi_rle_histogram_u8, rle_out)):
        src = db if name.endswith("dev") else hb
        for tag, args, expect in (
                ("null handle", (None, src, 1024, seg, 2, dst), INVALID),
                ("null hist", (ctx, src, 1024, seg, 2, None), INVALID),
                ("0 blocks", (ctx, src, 1024, seg, 0, dst), INVALID),
                ("65536 blocks", (ctx, src, 1024, seg, 65536, dst), INVALID),
                ("misaligned blocks", (ctx, src, 1000, 500, 2, dst), INVALID),
                ("blocks do not cover n", (ctx, src, 2048, seg, 2, dst), INVALID),
                ("a block past n", (ctx, src, 500, seg, 2, dst), INVALID),
                ("null grid", (ctx, None, 1024, seg, 2, dst), INVALID),
                ("empty, null grid", (ctx, None, 0, 0, 1, dst), 0),
                ("one block, any block_bytes", (ctx, src, 1000, 3, 1, dst), 0),
                ("two blocks", (ctx, src, 1000, seg, 2, dst), 0)):
            case((name, tag), f(*args), expect)
    bad_cases = {k: (got[k], want[k]) for k in want if got[k] != want[k]}
    assert not bad_cases, bad_cases


def _delta(L, handles, fn):
    """(kernel launches, graph launches) that `fn` adds to each context of `handles`."""
    before = [(L.hgi_ctx_kernel_launches(h), L.hgi_ctx_graph_launches(h)) for h in handles]
    rc = fn()
    assert rc == 0, rc
    after = [(L.hgi_ctx_kernel_launches(h), L.hgi_ctx_graph_launches(h)) for h in handles]
    return (tuple(a[0] - b[0] for a, b in zip(after, before)), tuple(a[1] - b[1] for a, b in zip(after, before)))


def test_launch_counts(env):
    import torch
    L, ctxs, pool, host, hout, dev, dout, dhist = env
    ctx, plv, gen = ctxs[hgi.PATH_TILE]._h, ctxs[hgi.PATH_PER_LEVEL]._h, ctxs[hgi.PATH_TILE_GENERIC]._h
    members = [L.hgi_pool_ctx(pool._h, k) for k in range(2)]
    hb, ho, db, do, dh = host.ctypes.data, hout.ctypes.data, dev.data_ptr(), dout.data_ptr(), dhist.data_ptr()
    keep = [np.zeros(N * 256, np.uint32), np.zeros(4 * 288, np.uint32), np.zeros(256, np.uint64)]
    keep += [np.zeros(1, np.uint64) for _ in range(3)]
    hh, rle_out, hist64, *mp = [a.ctypes.data for a in keep]
    rect = ctypes.byref(hgi._lib.RectStruct(0, 0, 10, 10))
    bands_in = ctypes.cast((ctypes.c_void_p * 2)(db, db), ctypes.c_void_p)
    bands_out = ctypes.cast((ctypes.c_void_p * 2)(do, do + 8192), ctypes.c_void_p)
    cases = [
        ("encode_u8", [ctx], lambda: L.hgi_encode_u8(ctx, hb, W, H, prm(), ho, None), 1),
        ("encode_u8 + recon", [ctx], lambda: L.hgi_encode_u8(ctx, hb, W, H, prm(), ho, ho + 4096), 1),
        ("decode_u8", [ctx], lambda: L.hgi_decode_u8(ctx, hb, W, H, prm(), ho), 1),
        ("encode_batch_u8 + hist", [ctx], lambda: L.hgi_encode_batch_u8(ctx, hb, N, W, H, prm(), ho, hh), 2),
        ("encode_batch_u8 L6", [ctx], lambda: L.hgi_encode_batch_u8(ctx, hb, N, W, H, prm(6), ho, None), 3),
        ("decode_batch_u8", [ctx], lambda: L.hgi_decode_batch_u8(ctx, hb, N, W, H, prm(), ho), 1),
        ("encode_dev + hist", [ctx], lambda: L.hgi_encode_dev(ctx, db, N, W, H, prm(), do, None, dh, None), 2),
        ("encode_dev L0", [ctx], lambda: L.hgi_encode_dev(ctx, db, N, W, H, prm(0), do, None, None, None), 0),
        ("encode_dev L0 + hist", [ctx], lambda: L.hgi_encode_dev(ctx, db, N, W, H, prm(0), do, None, dh, None), 1),
        ("decode_dev", [ctx], lambda: L.hgi_decode_dev(ctx, db, N, W, H, prm(), do, None), 1),
        ("encode_dev_pitched + hist", [ctx], lambda: L.hgi_encode_dev_pitched(ctx, db, N, W, H, 80, prm(), do, None, dh, None), 2),
        ("decode_dev_pitched", [ctx], lambda: L.hgi_decode_dev_pitched(ctx, db, N, W, H, 80, prm(), do, None), 1),
        ("histogram_dev", [ctx], lambda: L.hgi_histogram_dev(ctx, db, W * H, N, dh, None), 1),
        ("histogram_dev, empty planes", [ctx], lambda: L.hgi_histogram_dev(ctx, db, 0, N, dh, None), 0),
        ("histogram_u8", [ctx], lambda: L.hgi_histogram_u8(ctx, hb, 1000, hist64), 1),
        ("rle_histogram_dev", [ctx], lambda: L.hgi_rle_histogram_dev(ctx, db, 1000, 512, 2, dh, None), 1),
        ("rle_histogram_dev, empty", [ctx], lambda: L.hgi_rle_histogram_dev(ctx, db, 0, 0, 1, dh, None), 0),
        ("rle_histogram_u8", [ctx], lambda: L.hgi_rle_histogram_u8(ctx, hb, 1000, 512, 2, rle_out), 1),
        ("rle_histogram_u8, empty", [ctx], lambda: L.hgi_rle_histogram_u8(ctx, hb, 0, 0, 1, rle_out), 0),
        ("error_metrics_dev", [ctx], lambda: L.hgi_error_metrics_dev(ctx, db, db + 1, 1000, dh, None), 1),
        ("error_metrics_dev, empty", [ctx], lambda: L.hgi_error_metrics_dev(ctx, db, db, 0, dh, None), 0),
        ("error_metrics_u8", [ctx], lambda: L.hgi_error_metrics_u8(ctx, hb, hb + 1, 1000, *mp), 1),
        ("rgb_to_luma_dev", [ctx], lambda: L.hgi_rgb_to_luma_dev(ctx, db, 1000, do, None), 1),
        ("rgb_to_luma_u8", [ctx], lambda: L.hgi_rgb_to_luma_u8(ctx, hb, 1000, ho), 1),
        ("region_dev, scale 1", [ctx], lambda: L.hgi_decode_region_dev(ctx, db, N, W, H, W, prm(), 1, None, do, 32, None), 3),
        ("region_dev, rectangle", [ctx], lambda: L.hgi_decode_region_dev(ctx, db, N, W, H, W, prm(), 0, rect, do, 10, None), 3),
        ("region_dev, scale 4", [ctx], lambda: L.hgi_decode_region_dev(ctx, db, N, W, H, W, prm(), 4, None, do, 4, None), 2),
        ("region_dev, whole plane", [ctx], lambda: L.hgi_decode_region_dev(ctx, db, N, W, H, W, prm(), 0, None, do, W, None), 1),
        ("region_u8, scale 1", [ctx], lambda: L.hgi_decode_region_u8(ctx, hb, W, H, prm(), 1, None, ho), 3),
        # paths 1 and 2 run what path 0 runs
        ("path 1 encode_u8", [plv], lambda: L.hgi_encode_u8(plv, hb, W, H, prm(), ho, None), 1),
        ("path 1 decode_batch_u8", [plv], lambda: L.hgi_decode_batch_u8(plv, hb, N, W, H, prm(), ho), 1),
        ("path 2 encode_u8 L6", [gen], lambda: L.hgi_encode_u8(gen, hb, W, H, prm(6), ho, None), 3),
        ("pool encode_batch_u8 + hist", members, lambda: L.hgi_pool_encode_batch_u8(pool._h, hb, N, W, H, prm(), ho, hh), 2),
        ("pool decode_batch_u8", members, lambda: L.hgi_pool_decode_batch_u8(pool._h, hb, N, W, H, prm(), ho), 1),
        ("pool encode_plane_u8", members, lambda: L.hgi_pool_encode_plane_u8(pool._h, hb, W, H, prm(), ho), 1),
        ("pool decode_plane_u8", members, lambda: L.hgi_pool_decode_plane_u8(pool._h, hb, W, H, prm(), ho), 1),
        ("pool encode_bands_dev", members, lambda: L.hgi_pool_encode_bands_dev(pool._h, bands_in, W, H, prm(), bands_out), 1),
        ("pool decode_bands_dev", members, lambda: L.hgi_pool_decode_bands_dev(pool._h, bands_in, W, H, prm(), bands_out), 1),
    ]
    got, want = {}, {}
    for tag, cs, fn, n in cases:
        got[tag] = _delta(L, cs, fn)[0]
        torch.cuda.synchronize()
        want[tag] = tuple(n for _ in cs)
    # launch chains of the device API: run plainly, then captured, then replayed -- each call counts its kernels once
    for tag, c, lv, n in (("encode_dev L6 + hist", ctx, 6, 4), ("path 1 encode_dev L6 + hist", plv, 6, 4)):
        fn = (lambda c=c, lv=lv: L.hgi_encode_dev(c, db, N, W, H, prm(lv), do, None, dh, None))
        got[tag] = tuple(_delta(L, [c], fn) for _ in range(3))
        want[tag] = (((n,), (0,)), ((n,), (1,)), ((n,), (1,)))
    torch.cuda.synchronize()
    bad_cases = {k: (got[k], want[k]) for k in want if got[k] != want[k]}
    assert not bad_cases, bad_cases
    # the tile path's counts are the plain statement of its dispatch
    assert expected_launches("enc", 1, W, H, True, 6, N, hist=True) == 4
    assert expected_launches("enc", 1, W, H, True, 4, N, hist=True) == 2
