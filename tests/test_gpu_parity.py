"""Parity of the CUDA path (through the C ABI) with the oracle -- runs on the GPU box (-m gpu).

Bit-exact on grid bytes, reconstruction and decoded pixels for every golden config, both
interpolators, all quantizers, ragged and degenerate sizes, batches, the device-pointer API, histograms
and the `hgi test` metrics; every hgi_path_t value runs the same kernels.  Nothing here reads
/root/reference."""
import ctypes
import io

import numpy as np
import pytest

import rustyhgi_b200 as hgi
from conftest import get_plane, photo_like, sha16
from oracle import c as oc

pytestmark = pytest.mark.gpu

Q = hgi.QuantizationLevel


@pytest.fixture(scope="module")
def ctxs():
    # one context per hgi_path_t value: each runs the tile path, and the tests that take a path pin that it gives the
    # oracle's bytes whichever value a caller has set
    tile = hgi.Context(0, hgi.PATH_TILE)
    lvl = hgi.Context(0, hgi.PATH_PER_LEVEL)
    gen = hgi.Context(0, hgi.PATH_TILE_GENERIC)
    pre = hgi.Context(0, hgi.PATH_TILE_TMA)
    yield {"tile": tile, "level": lvl, "generic": gen, "tma": pre}
    for c in (tile, lvl, gen, pre):
        c.close()


def interp_of(i):
    return hgi.Crossed if i == oc.INTERP_CROSSED else hgi.LeftTop


def check_case(ctx, img, levels, q, interp=oc.INTERP_CROSSED, qkind=oc.QUANT_LINEAR):
    quant = hgi.Linear(Q(q)) if qkind == oc.QUANT_LINEAR else hgi.NoOp(Q(q))
    want_g, want_r = oc.encode(img, levels, interp=interp, qkind=qkind, qlevel=q, want_recon=True)
    enc = hgi.Encoder(interp_of(interp), quant, levels, ctx=ctx)
    grid, recon = enc.encode(img, want_recon=True)
    h, w = img.shape
    bad_g = int((grid.as_plane() != want_g).sum()) if img.size else 0
    bad_r = int((recon != want_r).sum())
    assert bad_g == 0 and bad_r == 0, f"{w}x{h} L{levels} q{q} i{interp}: grid {bad_g} recon {bad_r} bytes differ"
    grid_only = enc.encode(img)
    assert grid_only == grid
    dec = hgi.Decoder(interp_of(interp), ctx=ctx).decode((w, h), levels, grid)
    assert int((dec != want_r).sum()) == 0
    return grid, dec


@pytest.mark.parametrize("path", ["tile", "level", "generic"])
def test_reference_unit_fixture_all_levels(ctxs, path):
    """src/lib.rs:45-97 `test_error` on the 12x8 (x*y) image at levels=3 -- with the comparison
    against the *source* image that the reference's shadowed variable prevented."""
    img = get_plane("unit_12x8")
    for q in Q:
        quant = hgi.Linear.from_level(q)
        grid = hgi.Encoder(hgi.Crossed, quant, 3, ctx=ctxs[path]).encode(img)
        image = hgi.Decoder(hgi.Crossed, ctx=ctxs[path]).decode((12, 8), 3, grid)
        assert int(np.abs(img.astype(int) - image.astype(int)).max()) <= quant.error()
        assert (grid.as_plane() == oc.encode(img, 3, qlevel=int(q))).all()


@pytest.mark.parametrize("path", ["tile", "level", "generic"])
def test_golden_cases(ctxs, golden, path):
    for cs in golden["cases"]:
        img = get_plane(cs["plane"])
        grid, dec = check_case(ctxs[path], img, cs["levels"], cs["qlevel"], interp=cs["interp"])
        assert sha16(grid.as_plane()) == cs["grid_sha"] and sha16(dec) == cs["recon_sha"], cs
        m = hgi.error_metrics(img, dec, ctx=ctxs[path])
        assert (m["sd_int"], m["sum_sq"], m["max_abs"]) == (cs["sd_int"], cs["sum_sq"], cs["max_err"])


SIZES = [(1, 1), (1, 9), (9, 1), (2, 2), (3, 5), (16, 16), (17, 17), (127, 63), (128, 64), (129, 65), (130, 67),
         (144, 80), (145, 81), (250, 243), (256, 128), (257, 129), (272, 144), (300, 70), (1000, 3), (5, 700)]


@pytest.mark.parametrize("path", ["tile", "level", "generic"])
@pytest.mark.parametrize("w,h", SIZES)
def test_ragged_sizes(ctxs, path, w, h):
    img = photo_like(w, h, seed=w * 1000 + h)
    for levels, q in [(1, 1), (2, 3), (3, 2), (4, 2), (5, 1), (7, 3), (9, 2)]:
        check_case(ctxs[path], img, levels, q)
    check_case(ctxs[path], img, 4, 2, interp=oc.INTERP_LEFTTOP)
    check_case(ctxs[path], img, 6, 0, qkind=oc.QUANT_NOOP)


@pytest.mark.parametrize("path", ["tile", "level", "generic"])
def test_level_extremes(ctxs, path):
    img = photo_like(200, 120, 4)
    for levels in (0, 8, 12, 20, 30):
        check_case(ctxs[path], img, levels, 2)
    rnd = np.random.default_rng(5).integers(0, 256, (97, 211)).astype(np.uint8)   # worst case for fix-ups
    for q in range(4):
        check_case(ctxs[path], rnd, 4, q)
        check_case(ctxs[path], rnd, 5, q, interp=oc.INTERP_LEFTTOP)
    sat = np.where(np.indices((64, 160)).sum(0) % 2 == 0, 0, 255).astype(np.uint8)  # wrap-around extremes
    for q in range(4):
        check_case(ctxs[path], sat, 4, q)


@pytest.mark.parametrize("path", ["tile", "level", "generic"])
def test_aligned_multi_tile_planes(ctxs, path):
    """Widths that take the 128-bit path, several tiles in x and y, two passes (L > 4)."""
    for (w, h, levels, q) in [(512, 256, 4, 2), (640, 200, 6, 3), (1024, 520, 8, 1), (400, 400, 4, 1),
                              (128, 64, 4, 3), (144, 65, 3, 2), (272, 129, 2, 1), (1920, 1080, 1, 2), (2048, 70, 5, 3),
                              (16, 2000, 4, 2), (384, 384, 7, 0)]:
        img = photo_like(w, h, w + h)
        check_case(ctxs[path], img, levels, q)
        check_case(ctxs[path], img, levels, q, interp=oc.INTERP_LEFTTOP)
    rnd = np.random.default_rng(8).integers(0, 256, (200, 656)).astype(np.uint8)
    for q in range(4):
        for levels in (1, 2, 3, 4, 6):
            check_case(ctxs[path], rnd, levels, q)


def test_interior_and_edge_tile_split(ctxs):
    """The SWAR kernel runs interior tiles (tile + 17-pixel halo inside the plane) through a predicate-free body --
    a branch for the light kernels, launches of their own (interior / right tile columns / bottom tile rows) for the quantizing encode once the job has >= 5920 tiles.
    Sizes on either side of every boundary: no interior tile, one, an interior column without an interior row."""
    ctx = ctxs["tile"]
    for w in (144, 160, 272, 288, 400):           # 128-wide tiles: interior columns = (w - 17) // 128
        for h in (80, 81, 82, 144, 145, 146, 210):   # 64-high tiles: interior rows = (h - 17) // 64
            img = photo_like(w, h, seed=3 * w + h)
            for q in (0, 2, 3):
                check_case(ctx, img, 4, q)
            check_case(ctx, img, 4, 1, interp=oc.INTERP_LEFTTOP)
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    for (w, h) in [(144, 81), (160, 80), (160, 81), (272, 145), (288, 146), (416, 209), (256, 145), (384, 146), (128, 200)]:
        tiles = -(-w // 128) * -(-h // 64)
        n = -(-5920 // tiles) + 3                  # enough tiles for the two-launch path
        base = np.stack([photo_like(w, h, seed=s + w) for s in range(6)] +
                        [np.random.default_rng(w + h).integers(0, 256, (h, w)).astype(np.uint8)])
        imgs = base[np.arange(n) % len(base)]
        for q in (1, 3):
            enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), 4, ctx=ctx)
            launches0 = ctx.kernel_launches
            grids, hist = enc.encode_batch(imgs, want_hist=True)
            interior = ((w - 17) // 128) * ((h - 17) // 64) > 0
            # [interior + right tile columns +] bottom tile rows + histogram (a right column that is exactly one tile
            # wide -- w % 128 == 0 -- runs the body specialised for it)
            assert ctx.kernel_launches - launches0 == (4 if interior else 2), (w, h)
            want = oc.encode_batch(imgs[:len(base)], 4, qlevel=q)
            assert (grids == want[np.arange(n) % len(base)]).all(), (w, h, q)
            assert (hist[n - 1] == np.bincount(want[(n - 1) % len(base)].reshape(-1), minlength=256)).all()
            assert (dec.decode_batch(4, grids[-len(base):]) == oc.decode_batch(grids[-len(base):], 4)).all()
    launches0 = ctx.kernel_launches
    hgi.Encoder(hgi.Crossed, hgi.Linear(Q.Medium), 4, ctx=ctx).encode(imgs[0])
    assert ctx.kernel_launches - launches0 == 1    # a small job stays one launch


def test_batch_host_api_and_histograms(ctxs):
    ctx = ctxs["tile"]
    for (n, w, h, levels, q) in [(5, 160, 90, 4, 2), (3, 131, 77, 5, 3), (70, 256, 128, 4, 1)]:
        imgs = np.stack([photo_like(w, h, s + 1) for s in range(n)])
        enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels, ctx=ctx)
        grids, hist = enc.encode_batch(imgs, want_hist=True)
        want = oc.encode_batch(imgs, levels, qlevel=q)
        assert (grids == want).all()
        for i in range(n):
            assert (hist[i] == np.bincount(want[i].reshape(-1), minlength=256)).all()
        back = hgi.Decoder(hgi.Crossed, ctx=ctx).decode_batch(levels, grids)
        assert (back == oc.decode_batch(want, levels)).all()
        lv = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels, ctx=ctxs["level"]).encode_batch(imgs, want_hist=True)
        assert (lv[0] == want).all() and (lv[1] == hist).all()


def test_histogram_entry_point(ctxs):
    rng = np.random.default_rng(3)
    for n in (0, 1, 15, 16, 17, 1000, 65536, 1_000_003):
        data = (rng.integers(0, 256, n) * (rng.random(n) < 0.3)).astype(np.uint8)
        got = hgi.histogram(data, ctx=ctxs["tile"])
        assert (got == np.bincount(data, minlength=256)).all()
    off = np.zeros(4099, np.uint8)[3:]                      # unaligned base pointer
    off[:] = 7
    assert hgi.histogram(off, ctx=ctxs["tile"])[7] == 4096


def test_device_api_with_torch(ctxs):
    import torch
    ctx = ctxs["tile"]
    imgs = np.stack([get_plane("bench_1080p"), photo_like(1920, 1080, 2), photo_like(1920, 1080, 3)])
    t = torch.from_numpy(imgs).cuda()
    for q in (Q.Lossless, Q.Medium):
        enc = hgi.Encoder(hgi.Crossed, hgi.Linear(q), 4, ctx=ctx)
        hist = torch.empty((3, 256), dtype=torch.int32, device="cuda")
        recon = torch.empty_like(t)
        grids = enc.encode_device(t, recon_out=recon, hist_out=hist)
        dec = hgi.Decoder(hgi.Crossed, ctx=ctx).decode_device(4, grids)
        torch.cuda.synchronize()
        want_g = oc.encode_batch(imgs, 4, qlevel=int(q))
        want_r = oc.decode_batch(want_g, 4)
        assert (grids.cpu().numpy() == want_g).all()
        assert (dec.cpu().numpy() == want_r).all() and (recon.cpu().numpy() == want_r).all()
        assert (hist.cpu().numpy()[1] == np.bincount(want_g[1].reshape(-1), minlength=256)).all()
        assert (t.cpu().numpy() == imgs).all()              # input is const (reference consumes a copy)


def test_device_api_misaligned_bases_and_odd_widths(ctxs):
    """Planes whose base address and rows are not 16- (or even 4-) byte aligned take the funnel-shift / byte
    paths of the SWAR kernel; input, grid and image live at odd offsets inside larger allocations whose guard
    bytes must stay untouched."""
    import torch
    ctx = ctxs["tile"]
    for (n, h, w, levels, q) in [(2, 70, 160, 4, 2), (3, 65, 131, 3, 1), (1, 129, 255, 5, 3), (2, 64, 128, 4, 0)]:
        imgs = np.stack([photo_like(w, h, 7 * k + w) for k in range(n)])
        want_g = oc.encode_batch(imgs, levels, qlevel=q)
        want_r = oc.decode_batch(want_g, levels)
        for off in (1, 2, 3, 5):
            size = n * h * w
            src = torch.full((size + 64,), 0xAB, dtype=torch.uint8, device="cuda")
            dst = torch.full((size + 64,), 0xCD, dtype=torch.uint8, device="cuda")
            out = torch.full((size + 64,), 0xEF, dtype=torch.uint8, device="cuda")
            src[off:off + size] = torch.from_numpy(imgs).cuda().reshape(-1)
            s_v, d_v, o_v = (t[off:off + size].view(n, h, w) for t in (src, dst, out))
            enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels, ctx=ctx)
            enc.encode_device(s_v, grids_out=d_v)
            hgi.Decoder(hgi.Crossed, ctx=ctx).decode_device(levels, d_v, images_out=o_v)
            torch.cuda.synchronize()
            assert (d_v.cpu().numpy() == want_g).all() and (o_v.cpu().numpy() == want_r).all()
            for t, fill in ((dst, 0xCD), (out, 0xEF)):          # nothing written outside the planes
                assert bool((t[:off] == fill).all()) and bool((t[off + size:] == fill).all())


@pytest.mark.parametrize("path", ["tile", "level", "generic", "tma"])
def test_random_cases(ctxs, path):
    """Seeded random sweep over sizes (aligned and ragged), levels, quantizers, interpolators and image
    statistics: every byte of grid, reconstruction and decoded image must equal the oracle, on every hgi_path_t value,
    with as many kernels as HGI_PATH_TILE launches for the same calls."""
    rng = np.random.default_rng(20261018)
    kinds = ("noise", "smooth", "const", "extremes", "ramp")
    for case in range(70):
        w = int(rng.choice([16, 32, 48, 128, 144, 160, 256, 272, 400])) if case % 2 == 0 else int(rng.integers(1, 420))
        h = int(rng.integers(1, 300))
        levels = int(rng.integers(0, 10))
        q = int(rng.integers(0, 4))
        interp = oc.INTERP_CROSSED if rng.random() < 0.8 else oc.INTERP_LEFTTOP
        kind = kinds[case % len(kinds)]
        if kind == "noise":
            img = rng.integers(0, 256, (h, w)).astype(np.uint8)
        elif kind == "smooth":
            img = photo_like(w, h, case)
        elif kind == "const":
            img = np.full((h, w), int(rng.integers(0, 256)), np.uint8)
        elif kind == "extremes":
            img = (rng.integers(0, 2, (h, w)) * 255).astype(np.uint8)
        else:
            yy, xx = np.mgrid[0:h, 0:w]
            img = ((xx * 5 + yy * 3) & 255).astype(np.uint8)
        ctx, ref = ctxs[path], ctxs["tile"]
        launches = ctx.kernel_launches
        check_case(ctx, img, levels, q, interp=interp)
        launches = ctx.kernel_launches - launches
        if ctx is not ref:
            want = ref.kernel_launches
            check_case(ref, img, levels, q, interp=interp)
            assert launches == ref.kernel_launches - want, (case, w, h, levels)


def test_more_images_than_grid_z(ctxs):
    """A batch larger than gridDim.z (65535) is cut into several launches of the SWAR kernel."""
    import torch
    n, h, w = 66000, 16, 16
    rng = np.random.default_rng(11)
    imgs = rng.integers(0, 256, (n, h, w)).astype(np.uint8)
    t = torch.from_numpy(imgs).cuda()
    enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Q.High), 3, ctx=ctxs["tile"])
    grids = enc.encode_device(t)
    back = hgi.Decoder(hgi.Crossed, ctx=ctxs["tile"]).decode_device(3, grids)
    torch.cuda.synchronize()
    g = grids.cpu().numpy()
    for i in (0, 1, 65534, 65535, 65536, n - 1):
        want = oc.encode(imgs[i], 3, qlevel=3)
        assert (g[i] == want).all()
        assert (back[i].cpu().numpy() == oc.decode(want, 3)).all()
    assert int((back.to(torch.int16) - t.to(torch.int16)).abs().max().item()) <= 30


def test_archive_roundtrip_from_gpu_grid(ctxs):
    """`hgi test`-style flow (src/main.rs:73-120) on LENA.TIF level 4 Medium = BASELINE config 1."""
    img = get_plane("lena_tif")
    grid = hgi.Encoder(hgi.Crossed, hgi.Linear(Q.Medium), 4, ctx=ctxs["tile"]).encode(img)
    md = hgi.Metadata(Q.Medium, hgi.InterpolationType.Crossed, 256, 256, 4)
    buf = io.BytesIO()
    hgi.Archive(md, grid).serialize_to_writer(buf)
    arch = hgi.Archive.deserialize_from_reader(io.BytesIO(buf.getvalue()))
    after = hgi.Decoder(hgi.Crossed, ctx=ctxs["tile"]).decode((arch.metadata.width, arch.metadata.height),
                                                              arch.metadata.scale_level, arch.grid)
    m = hgi.error_metrics(img, after, ctx=ctxs["tile"])
    assert img.size // 1024 == 64 and f"{m['sd']:.2f}" == "9.17"
    assert sha16(after) == "e17f5ad9f400234e" and sha16(grid.as_plane()) == "3a992020370c96a4"


def test_unsupported_and_invalid(ctxs):
    L = hgi.lib()
    buf = np.zeros(64, np.uint8)
    for interp, want in ((1, -8), (2, -8), (9, -1)):
        p = hgi._lib.Params(3, interp, 1, 2)
        assert L.hgi_encode_u8(ctxs["tile"]._h, buf.ctypes.data, 8, 8, ctypes.byref(p), buf.ctypes.data, None) == want
    p = hgi._lib.Params(32, 0, 1, 2)
    assert L.hgi_encode_u8(ctxs["tile"]._h, buf.ctypes.data, 8, 8, ctypes.byref(p), buf.ctypes.data, None) == -1
    p = hgi._lib.Params(3, 0, 1, 2)
    assert L.hgi_encode_u8(ctxs["tile"]._h, None, 8, 8, ctypes.byref(p), buf.ctypes.data, None) == -1
    assert L.hgi_encode_u8(ctxs["tile"]._h, buf.ctypes.data, 0, 8, ctypes.byref(p), buf.ctypes.data, None) == 0
