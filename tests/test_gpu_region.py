"""Scalable decode on the B200 (-m gpu): hgi_decode_region_dev / hgi_decode_region_u8 against the oracle's full
decode, decimated by 2^k and sliced, on the golden planes, ragged sizes, padded batches, several streams and the
16384^2 level-8 plane; argument errors; the CLI's --scale / --region."""
import ctypes
import os

import numpy as np
import pytest

import rustyhgi_b200 as hgi
from conftest import get_plane, photo_like
from oracle import c as oc
from rustyhgi_b200 import cli

pytestmark = pytest.mark.gpu
PATHS = {"tile": hgi.PATH_TILE}
INTERPS = {"crossed": (hgi.Crossed, oc.INTERP_CROSSED), "lefttop": (hgi.LeftTop, oc.INTERP_LEFTTOP)}


@pytest.fixture(scope="module")
def contexts():
    ctxs = {name: hgi.Context(0, path=p) for name, p in PATHS.items()}
    yield ctxs
    for c in ctxs.values():
        c.close()


def scaled_size(w, h, k):
    return -(-w // (1 << k)), -(-h // (1 << k))


def regions(ws, hs):
    """whole; 1x1 at the origin and at the last pixel; an odd interior rectangle; rectangles touching the right and
    the bottom edge; a full row; a full column."""
    def clip(x, y, w, h):
        x, y = min(x, ws - 1), min(y, hs - 1)
        return (x, y, max(1, min(w, ws - x)), max(1, min(h, hs - y)))
    out = [None, (0, 0, 1, 1), (ws - 1, hs - 1, 1, 1), clip(ws // 7 + 1, hs // 5 + 1, (ws // 2) | 1, (hs // 3) | 1),
           clip(ws - min(ws, 37), hs // 3, 37, (hs // 4) | 1), clip(ws // 5, hs - min(hs, 23), (ws // 3) | 1, 23),
           (0, hs // 2, ws, 1), (ws // 2, 0, 1, hs)]
    return list(dict.fromkeys(out))


def cut(full, k, region):
    s = full[::1 << k, ::1 << k]
    if region is None:
        return s
    x, y, w, h = region
    return s[y:y + h, x:x + w]


GOLDEN = [("lena_tif", 4), ("docs_lena_source", 4), ("fullhd", 4), ("ikonos", 6), ("bench_1080p", 4)]


@pytest.mark.parametrize("plane,levels", GOLDEN)
@pytest.mark.parametrize("interp", list(INTERPS))
def test_golden_planes_every_scale_region_and_path(contexts, plane, levels, interp):
    import torch
    cls, oid = INTERPS[interp]
    img = get_plane(plane)
    h, w = img.shape
    grid = oc.encode(img, levels, interp=oid, qlevel=oc.MEDIUM)
    full = oc.decode(grid, levels, interp=oid)
    g = torch.from_numpy(grid).cuda()
    for name, ctx in contexts.items():
        dec = hgi.Decoder(cls, ctx=ctx)
        for k in range(levels + 2):
            for region in regions(*scaled_size(w, h, k)):
                got = dec.decode_region_device(levels, g, region=region, scale_log2=k)
                assert np.array_equal(got.cpu().numpy(), cut(full, k, region)), (name, k, region)


def test_ragged_sizes_and_deep_hierarchies():
    """Widths 1, 15, 17, 1919, heights 1, 65 and seeded ones, L up to 12 (windows that need several passes); the host
    entry point and the device entry point."""
    import torch
    rng = np.random.default_rng(2024)
    sizes = [(1, 1), (15, 65), (17, 1), (1919, 65), (1, 300), (1919, 1)]
    sizes += [(int(rng.integers(1, 2100)), int(rng.integers(1, 700))) for _ in range(34)]
    for i, (w, h) in enumerate(sizes):
        levels = int(rng.integers(0, 13))
        k = int(rng.integers(0, levels + 2))
        cls, oid = list(INTERPS.values())[i % 2]
        img = photo_like(w, h, i)
        grid = oc.encode(img, levels, interp=oid, qlevel=i % 4)
        full = oc.decode(grid, levels, interp=oid)
        ws, hs = scaled_size(w, h, k)
        x, y = int(rng.integers(0, ws)), int(rng.integers(0, hs))
        region = (x, y, int(rng.integers(1, ws - x + 1)), int(rng.integers(1, hs - y + 1)))
        dec = hgi.Decoder(cls)
        want = cut(full, k, region)
        assert np.array_equal(dec.decode_region((w, h), levels, grid, region, k), want), (w, h, levels, k, region)
        got = dec.decode_region_device(levels, torch.from_numpy(grid).cuda(), region=region, scale_log2=k)
        assert np.array_equal(got.cpu().numpy(), want), (w, h, levels, k, region)


def padded_batch(n=5, w=1919, h=301, pitch=2048, levels=6):
    import torch
    frames = np.stack([photo_like(w, h, 40 + i) for i in range(n)])
    grids = oc.encode_batch(frames, levels, qlevel=oc.MEDIUM)
    fulls = oc.decode_batch(grids, levels)
    buf = torch.randint(0, 256, (n, h, pitch), dtype=torch.uint8, device="cuda")   # garbage in the padding
    buf[..., :w] = torch.from_numpy(grids).cuda()
    return buf[..., :w], fulls


def test_batch_padded_input_and_output_rows_and_sentinels():
    import torch
    g, fulls = padded_batch()
    n, levels = g.shape[0], 6
    dec = hgi.Decoder(hgi.Crossed)
    for k, region in ((0, (13, 7, 501, 97)), (1, (3, 0, 957, 151)), (2, None), (3, (0, 5, 17, 1)), (0, None), (7, None)):
        ws, hs = scaled_size(1919, 301, k)
        rw, rh = (ws, hs) if region is None else region[2:]
        out_pitch, guard = ((rw + 40) | 1), 4096                       # odd pitch: no row starts 16-byte aligned
        flat = torch.full((2 * guard + n * rh * out_pitch,), 0xA5, dtype=torch.uint8, device="cuda")
        out = flat[guard:guard + n * rh * out_pitch].view(n, rh, out_pitch)[..., :rw]
        dec.decode_region_device(levels, g, region=region, scale_log2=k, out=out)
        torch.cuda.synchronize()
        for i in range(n):
            assert np.array_equal(out[i].cpu().numpy(), cut(fulls[i], k, region)), (k, region, i)
        mask = torch.ones_like(flat, dtype=torch.bool)
        mask[guard:guard + n * rh * out_pitch].view(n, rh, out_pitch)[..., :rw] = False
        assert bool((flat[mask] == 0xA5).all()), (k, region)              # padding and the guard bands untouched


def test_batch_on_a_side_stream_and_two_streams_at_once():
    import torch
    g, fulls = padded_batch()
    levels = 6
    ctx = hgi.Context(0)
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = dec.decode_region_device(levels, g, region=(100, 50, 700, 100), scale_log2=1, stream=s.cuda_stream)
    s.synchronize()
    for i in range(g.shape[0]):
        assert np.array_equal(got[i].cpu().numpy(), cut(fulls[i], 1, (100, 50, 700, 100)))
    # two streams of one context with different regions in flight together (each stream owns its scratch set)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    cases = [(s1, 0, (1000, 40, 900, 250)), (s2, 2, (5, 3, 400, 70))]
    outs = []
    for _ in range(3):
        for st, k, region in cases:
            with torch.cuda.stream(st):
                outs.append((k, region, dec.decode_region_device(levels, g, region=region, scale_log2=k, stream=st.cuda_stream)))
    s1.synchronize()
    s2.synchronize()
    for k, region, o in outs:
        for i in range(g.shape[0]):
            assert np.array_equal(o[i].cpu().numpy(), cut(fulls[i], k, region)), (k, region, i)
    ctx.close()


def test_config4_viewport_and_overviews():
    """16384^2, L8, Medium: a 1920x1080 viewport and overviews at k = 4 and 8 against the product's full decode
    (tests/test_gpu_fullsize.py checks that one against the oracle), with the launches each call costs."""
    import torch
    n = 16384
    x = torch.arange(n, device="cuda", dtype=torch.int32)
    img = ((x[None, :] * x[:, None]) & 255).to(torch.uint8).contiguous()
    ctx = hgi.Context(0)
    grid = hgi.Encoder(hgi.Crossed, hgi.Linear(hgi.QuantizationLevel.Medium), 8, ctx=ctx).encode_device(img)
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    full = dec.decode_device(8, grid)
    torch.cuda.synchronize()
    del img
    for k, region in ((0, (5000, 7000, 1920, 1080)), (4, None), (8, None)):
        before = ctx.kernel_launches
        got = dec.decode_region_device(8, grid, region=region, scale_log2=k)
        torch.cuda.synchronize()
        launches = ctx.kernel_launches - before
        s = full[::1 << k, ::1 << k]
        want = s if region is None else s[region[1]:region[1] + region[3], region[0]:region[0] + region[2]]
        assert torch.equal(got, want), (k, region)
        # gather + the window's passes (none at k = 8: the window of the grid is the image) + crop
        assert (launches == 2) if k == 8 else (3 <= launches <= 8), (k, launches)
    # the host entry point gives the same bytes as the device one
    host_grid = grid.cpu().numpy()
    for k, region in ((0, (5000, 7000, 1920, 1080)), (3, (100, 1500, 333, 17))):
        got = dec.decode_region((n, n), 8, host_grid, region, k)
        dev = dec.decode_region_device(8, grid, region=region, scale_log2=k)
        assert np.array_equal(got, dev.cpu().numpy()), (k, region)
    ctx.close()


def test_error_codes():
    import torch
    L = hgi.lib()
    ctx = hgi.Context(0)
    g = torch.zeros((64, 48), dtype=torch.uint8, device="cuda")
    o = torch.zeros((64, 48), dtype=torch.uint8, device="cuda")

    def dev(region=None, k=0, out_pitch=48, n=1, interp=0, ctx_h=ctx._h, grids=g.data_ptr(), out=o.data_ptr(), levels=4):
        p = hgi._lib.Params(levels, interp, 0, 0)
        r = ctypes.byref(hgi._lib.RectStruct(*region)) if region is not None else None
        return L.hgi_decode_region_dev(ctx_h, grids, n, 48, 64, 48, ctypes.byref(p), k, r, out, out_pitch, None)

    def host(region=None, k=0, interp=0):
        p = hgi._lib.Params(4, interp, 0, 0)
        r = ctypes.byref(hgi._lib.RectStruct(*region)) if region is not None else None
        buf = np.zeros(64 * 48, np.uint8)
        return L.hgi_decode_region_u8(ctx._h, buf.ctypes.data, 48, 64, ctypes.byref(p), k, r, buf.ctypes.data)

    assert dev() == 0 and dev((1, 2, 3, 4), 1, out_pitch=3) == 0 and host((0, 0, 24, 32), 1) == 0
    for region, k in (((0, 0, 0, 4), 0), ((0, 0, 4, 0), 0), ((0, 0, 25, 1), 1), ((47, 0, 2, 1), 0), ((0, 63, 1, 2), 0),
                      (None, 32)):
        assert dev(region, k) == -1 and host(region, k) == -1, (region, k)
    assert dev(levels=32) == -1
    assert dev((0, 0, 10, 10), out_pitch=9) == -1                       # out_pitch < region width
    assert dev(grids=None) == -1 and dev(out=None) == -1
    assert dev(n=0, grids=None, out=None) == 0                          # nothing to do
    assert dev(interp=1) == -8 and dev(interp=2) == -8 and host(interp=1) == -8   # Line / Previous
    assert dev(interp=7) == -1
    # every path value runs the tile path: regions on a PATH_PER_LEVEL context are the oracle's
    img = photo_like(48, 64, 9)
    grid = oc.encode(img, 4, qlevel=oc.MEDIUM)
    full = oc.decode(grid, 4)
    gg = torch.from_numpy(grid).cuda()
    per_level = hgi.Context(0, path=hgi.PATH_PER_LEVEL)
    for region, k in ((None, 0), ((0, 0, 5, 5), 2), ((3, 7, 9, 5), 1)):
        o.fill_(0x5A)
        assert dev(region, k, ctx_h=per_level._h, grids=gg.data_ptr()) == 0
        torch.cuda.synchronize()
        want = cut(full, k, region)
        assert np.array_equal(o.cpu().numpy()[:want.shape[0], :want.shape[1]], want), (region, k)
    per_level.close()
    with pytest.raises(hgi.HgiError):
        hgi.Decoder(hgi.Crossed, ctx=ctx).decode_region_device(4, g, region=(40, 0, 9, 1))
    ctx.close()


def test_cli_decode_scale_and_region_round_trip(tmp_path):
    from PIL import Image
    src = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fullhd.png")
    arc, whole, part = (str(tmp_path / f) for f in ("a.hgi", "whole.png", "part.png"))
    cli.main(["encode", "-i", src, "-o", arc, "-l", "4", "-q", "medium"])
    cli.main(["decode", "-i", arc, "-o", whole])
    cli.main(["decode", "-i", arc, "-o", part, "--scale", "2", "--region", "31,17,301,203"])
    full = np.array(Image.open(whole))
    got = np.array(Image.open(part))
    assert got.shape == (203, 301)
    assert np.array_equal(got, full[::4, ::4][17:17 + 203, 31:31 + 301])
