"""Batched crops on the B200 (-m gpu): hgi_decode_crops_dev against the oracle's full decode, decimated by 2^k and
sliced at each plane's own origin -- golden planes at every scale with both interpolators, 1080p frames
with random crops, padded rows, clamped origins, two streams, a caller's CUDA graph with origins rewritten in place,
more than 65 535 planes, launch counts and every error code."""
import ctypes

import numpy as np
import pytest

import rustyhgi_b200 as hgi
from conftest import get_plane, photo_like
from oracle import c as oc

pytestmark = pytest.mark.gpu
PATHS = {"tile": hgi.PATH_TILE}
INTERPS = {"crossed": (hgi.Crossed, oc.INTERP_CROSSED), "lefttop": (hgi.LeftTop, oc.INTERP_LEFTTOP)}


def scaled_size(w, h, k):
    return -(-w // (1 << k)), -(-h // (1 << k))


def want_crops(fulls, k, xy, cw, ch):
    """fulls: the oracle's full decodes (n, h, w) or one plane for all; xy: the clamped origins."""
    out = []
    for i, (x, y) in enumerate(xy):
        s = (fulls[i] if fulls.ndim == 3 else fulls)[::1 << k, ::1 << k]
        out.append(s[y:y + ch, x:x + cw])
    return np.stack(out)


def random_origins(rng, n, ws, hs, cw, ch):
    return np.stack([rng.integers(0, ws - cw + 1, n), rng.integers(0, hs - ch + 1, n)], axis=1).astype(np.int32)


def dev_origins(xy):
    import torch
    return torch.from_numpy(np.ascontiguousarray(xy, dtype=np.int32)).cuda()


@pytest.fixture(scope="module")
def contexts():
    ctxs = {name: hgi.Context(0, path=p) for name, p in PATHS.items()}
    yield ctxs
    for c in ctxs.values():
        c.close()


GOLDEN = [("lena_tif", 4), ("docs_lena_source", 4), ("fullhd", 4), ("ikonos", 6), ("bench_1080p", 4)]


@pytest.mark.parametrize("plane,levels", GOLDEN)
@pytest.mark.parametrize("interp", list(INTERPS))
def test_golden_planes_stacked_with_different_origins(contexts, plane, levels, interp):
    import torch
    cls, oid = INTERPS[interp]
    img = get_plane(plane)
    h, w = img.shape
    grid = oc.encode(img, levels, interp=oid, qlevel=oc.MEDIUM)
    full = oc.decode(grid, levels, interp=oid)
    n = 6
    g = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(grid, (n, h, w)))).cuda()
    rng = np.random.default_rng(len(plane) * 31 + levels)
    for name, ctx in contexts.items():
        dec = hgi.Decoder(cls, ctx=ctx)
        for k in range(levels + 2):
            ws, hs = scaled_size(w, h, k)
            for cw, ch in dict.fromkeys([(1, 1), (min(ws, 224), min(hs, 224)), ((ws // 3) | 1, (hs // 5) | 1), (ws, hs)]):
                xy = random_origins(rng, n, ws, hs, cw, ch)
                xy[0], xy[1] = (0, 0), (ws - cw, hs - ch)
                got = dec.decode_crops_device(levels, g, dev_origins(xy), (cw, ch), scale_log2=k)
                assert np.array_equal(got.cpu().numpy(), want_crops(full, k, xy, cw, ch)), (name, k, cw, ch)


def test_photo_frames_random_crops():
    """64 photo-like 1080p frames, L4 Medium, 224 x 224 crops at random origins, k = 0, 1, 2."""
    import torch
    n, w, h, levels = 64, 1920, 1080, 4
    frames = np.stack([photo_like(w, h, 300 + i) for i in range(n)])
    grids = oc.encode_batch(frames, levels, qlevel=oc.MEDIUM)
    fulls = oc.decode_batch(grids, levels)
    g = torch.from_numpy(grids).cuda()
    dec = hgi.Decoder(hgi.Crossed)
    rng = np.random.default_rng(5)
    for k in (0, 1, 2):
        ws, hs = scaled_size(w, h, k)
        xy = random_origins(rng, n, ws, hs, 224, 224)
        got = dec.decode_crops_device(levels, g, dev_origins(xy), (224, 224), scale_log2=k)
        assert np.array_equal(got.cpu().numpy(), want_crops(fulls, k, xy, 224, 224)), k


def padded_batch(n=5, w=1919, h=301, pitch=2048, levels=6):
    import torch
    frames = np.stack([photo_like(w, h, 60 + i) for i in range(n)])
    grids = oc.encode_batch(frames, levels, qlevel=oc.MEDIUM)
    fulls = oc.decode_batch(grids, levels)
    buf = torch.randint(0, 256, (n, h, pitch), dtype=torch.uint8, device="cuda")   # garbage in the padding
    buf[..., :w] = torch.from_numpy(grids).cuda()
    return buf[..., :w], fulls


def test_padded_input_rows_odd_out_pitch_and_sentinels():
    import torch
    g, fulls = padded_batch()
    n, levels = g.shape[0], 6
    dec = hgi.Decoder(hgi.Crossed)
    rng = np.random.default_rng(8)
    for k, (cw, ch) in ((0, (501, 97)), (1, (957, 151)), (2, (17, 1)), (3, (240, 38)), (7, (15, 3))):
        ws, hs = scaled_size(1919, 301, k)
        xy = random_origins(rng, n, ws, hs, cw, ch)
        out_pitch, guard = ((cw + 40) | 1), 4096                       # odd pitch: no row starts 16-byte aligned
        flat = torch.full((2 * guard + n * ch * out_pitch,), 0xA5, dtype=torch.uint8, device="cuda")
        out = flat[guard:guard + n * ch * out_pitch].view(n, ch, out_pitch)[..., :cw]
        dec.decode_crops_device(levels, g, dev_origins(xy), (cw, ch), scale_log2=k, out=out)
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), want_crops(fulls, k, xy, cw, ch)), (k, cw, ch)
        mask = torch.ones_like(flat, dtype=torch.bool)
        mask[guard:guard + n * ch * out_pitch].view(n, ch, out_pitch)[..., :cw] = False
        assert bool((flat[mask] == 0xA5).all()), (k, cw, ch)               # padding and the guard bands untouched


def test_origins_are_clamped_into_the_image():
    g, fulls = padded_batch()
    n, levels = g.shape[0], 6
    dec = hgi.Decoder(hgi.Crossed)
    big = 2**31 - 1
    raw = np.array([(-5, -5), (big, big), (-5, big), (big, -5), (-(2**31), 7)], np.int32)
    for k, (cw, ch) in ((0, (224, 224)), (2, (33, 20)), (9, (1, 1))):
        ws, hs = scaled_size(1919, 301, k)
        xy = np.stack([np.clip(raw[:, 0].astype(np.int64), 0, ws - cw), np.clip(raw[:, 1].astype(np.int64), 0, hs - ch)], 1)
        got = dec.decode_crops_device(levels, g, dev_origins(raw), (cw, ch), scale_log2=k)
        assert np.array_equal(got.cpu().numpy(), want_crops(fulls, k, xy, cw, ch)), k


def test_equal_origins_give_the_region_decode():
    import torch
    g, fulls = padded_batch()
    n, levels = g.shape[0], 6
    dec = hgi.Decoder(hgi.Crossed)
    for k, region in ((0, (13, 7, 501, 97)), (1, (3, 0, 957, 151)), (3, (200, 5, 17, 1))):
        xy = torch.tensor([region[:2]] * n, dtype=torch.int32, device="cuda")
        got = dec.decode_crops_device(levels, g, xy, region[2:], scale_log2=k)
        assert torch.equal(got, dec.decode_region_device(levels, g, region=region, scale_log2=k)), (k, region)


def test_two_streams_of_one_context_at_once():
    import torch
    g, fulls = padded_batch()
    n, levels = g.shape[0], 6
    ctx = hgi.Context(0)
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    rng = np.random.default_rng(9)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    cases = [(s1, 0, (900, 250)), (s2, 2, (400, 70))]
    outs = []
    for _ in range(3):
        for st, k, (cw, ch) in cases:
            xy = random_origins(rng, n, *scaled_size(1919, 301, k), cw, ch)
            o = dev_origins(xy)
            st.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(st):
                outs.append((k, xy, cw, ch, dec.decode_crops_device(levels, g, o, (cw, ch), scale_log2=k, stream=st.cuda_stream)))
                o.record_stream(st)
    s1.synchronize()
    s2.synchronize()
    for k, xy, cw, ch, o in outs:
        assert np.array_equal(o.cpu().numpy(), want_crops(fulls, k, xy, cw, ch)), (k, cw, ch)
    ctx.close()


def test_callers_cuda_graph_replays_with_new_origins():
    """One warm-up call sizes the scratch; the caller's own torch.cuda.graph capture then allocates nothing and syncs
    nothing, and each replay reads the origins written in place since."""
    import torch
    g, fulls = padded_batch()
    n, levels, k, cw, ch = g.shape[0], 6, 1, 300, 120
    ws, hs = scaled_size(1919, 301, k)
    ctx = hgi.Context(0)
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    rng = np.random.default_rng(10)
    origins = dev_origins(random_origins(rng, n, ws, hs, cw, ch))
    out = torch.empty((n, ch, cw), dtype=torch.uint8, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        dec.decode_crops_device(levels, g, origins, (cw, ch), scale_log2=k, out=out)      # warm-up: same shapes
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):                           # the warmed-up stream owns the sized scratch
        dec.decode_crops_device(levels, g, origins, (cw, ch), scale_log2=k, out=out)
    for _ in range(3):
        xy = random_origins(rng, n, ws, hs, cw, ch)
        origins.copy_(torch.from_numpy(xy))
        out.fill_(0)
        graph.replay()
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy(), want_crops(fulls, k, xy, cw, ch))
    del graph
    ctx.close()


def test_more_than_65535_planes():
    """70 000 planes of 40 x 24 (16 distinct ones, repeated), 8 x 8 crops: the copy kernels' grid-stride loops and the
    tile path past the 65 535-plane launch limit."""
    import torch
    n, w, h, levels = 70_000, 40, 24, 4
    base = np.stack([photo_like(w, h, 900 + i) for i in range(16)])
    grids = oc.encode_batch(base, levels, qlevel=oc.MEDIUM)
    fulls = oc.decode_batch(grids, levels)
    g = torch.from_numpy(grids).cuda().repeat(n // 16 + 1, 1, 1)[:n].contiguous()
    rng = np.random.default_rng(11)
    dec = hgi.Decoder(hgi.Crossed)
    for k in (0, 1):
        ws, hs = scaled_size(w, h, k)
        xy = random_origins(rng, n, ws, hs, 8, 8)
        got = dec.decode_crops_device(levels, g, dev_origins(xy), (8, 8), scale_log2=k).cpu().numpy()
        idx = np.arange(n) % 16
        for j in range(16):
            sel = idx == j
            assert np.array_equal(got[sel], want_crops(fulls[j], k, xy[sel], 8, 8)), (k, j)


def test_launch_counts():
    """gather + crop + the kernels of hgi_decode_dev_pitched on n planes of the window size with L' levels."""
    import torch
    L = hgi.lib()
    ctx = hgi.Context(0)
    n, w, h = 3, 1920, 1080
    g = torch.zeros((n, h, w), dtype=torch.uint8, device="cuda")
    out = torch.zeros(n * w * h, dtype=torch.uint8, device="cuda")
    org = torch.zeros((n, 2), dtype=torch.int32, device="cuda")
    for levels, k, (cw, ch) in ((4, 0, (224, 224)), (4, 1, (256, 256)), (4, 2, (128, 128)), (8, 0, (1000, 900)),
                                (4, 4, (100, 60)), (4, 6, (30, 16)), (9, 0, (1920, 1080))):
        dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
        before = ctx.kernel_launches
        dec.decode_crops_device(levels, g, org, (cw, ch), scale_log2=k)
        torch.cuda.synchronize()
        crops = ctx.kernel_launches - before
        pl = hgi.plan_crop(w, h, levels, k, (0, 0, cw, ch))
        dx, dy = pl.window[2:]
        pitch = -(-dx // 16) * 16
        p = hgi._lib.Params(pl.levels, 0, 0, 0)
        before = ctx.kernel_launches
        assert L.hgi_decode_dev_pitched(ctx._h, g.data_ptr(), n, dx, dy, pitch, ctypes.byref(p), out.data_ptr(), None) == 0
        torch.cuda.synchronize()
        window = ctx.kernel_launches - before
        assert crops == 2 + window, (levels, k, cw, ch, crops, window)
        if pl.levels == 0:
            assert crops == 2
    ctx.close()


def test_error_codes():
    import torch
    L = hgi.lib()
    ctx = hgi.Context(0)
    g = torch.zeros((2, 64, 48), dtype=torch.uint8, device="cuda")
    o = torch.zeros((2, 64, 48), dtype=torch.uint8, device="cuda")
    org = torch.zeros(8, dtype=torch.int32, device="cuda")

    def dev(cw=8, ch=8, k=0, out_pitch=48, n=2, interp=0, ctx_h=ctx._h, grids=g.data_ptr(), out=o.data_ptr(),
            origins=org.data_ptr(), levels=4):
        p = hgi._lib.Params(levels, interp, 0, 0)
        return L.hgi_decode_crops_dev(ctx_h, grids, n, 48, 64, 48, ctypes.byref(p), k, cw, ch, origins, out, out_pitch, None)

    assert dev() == 0 and dev(48, 64) == 0 and dev(24, 32, 1, out_pitch=24) == 0 and dev(1, 1, 31) == 0
    for cw, ch, k in ((0, 4, 0), (4, 0, 0), (49, 1, 0), (1, 65, 0), (25, 1, 1), (2, 1, 7), (1, 1, 32)):
        assert dev(cw, ch, k) == -1, (cw, ch, k)
    assert dev(levels=32) == -1
    assert dev(10, 10, out_pitch=9) == -1                              # out_pitch < crop width
    assert dev(grids=None) == -1 and dev(out=None) == -1 and dev(origins=None) == -1
    assert dev(origins=org.data_ptr() + 2) == -1                       # origins not 4-byte aligned
    assert dev(origins=org.data_ptr() + 4) == 0                        # 4-byte aligned is enough
    assert dev(n=0, grids=None, out=None, origins=None) == 0           # nothing to do
    assert dev(ctx_h=None) == -1
    assert dev(interp=1) == -8 and dev(interp=2) == -8                 # Line / Previous
    assert dev(interp=7) == -1
    # every path value runs the tile path: crops on a PATH_PER_LEVEL context are the oracle's
    imgs = np.stack([photo_like(48, 64, 9 + i) for i in range(2)])
    grids = oc.encode_batch(imgs, 4, qlevel=oc.MEDIUM)
    fulls = oc.decode_batch(grids, 4)
    gg = torch.from_numpy(grids).cuda()
    xy = np.array([[3, 5], [40, 60]], np.int32)          # the second origin is clamped
    d_xy = dev_origins(xy)
    per_level = hgi.Context(0, path=hgi.PATH_PER_LEVEL)
    for cw, ch, k in ((8, 8, 0), (5, 5, 2)):
        ws, hs = scaled_size(48, 64, k)
        clamped = np.minimum(xy, [ws - cw, hs - ch])
        o.fill_(0x5A)
        assert dev(cw, ch, k, ctx_h=per_level._h, grids=gg.data_ptr(), origins=d_xy.data_ptr()) == 0
        torch.cuda.synchronize()
        got = o.cpu().numpy().reshape(-1)[:2 * 48 * ch].reshape(2, ch, 48)[:, :, :cw]
        assert np.array_equal(got, want_crops(fulls, k, clamped, cw, ch)), (cw, ch, k)
    per_level.close()
    # n == 0 launches nothing
    before = ctx.kernel_launches
    assert dev(n=0) == 0
    assert ctx.kernel_launches == before
    # the Python layer
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    good = torch.zeros((2, 2), dtype=torch.int32, device="cuda")
    assert dec.decode_crops_device(4, g, good, (8, 8)).shape == (2, 8, 8)
    for bad in (good.to(torch.int64), good.cpu(), torch.zeros((3, 2), dtype=torch.int32, device="cuda"),
                torch.zeros((2, 3), dtype=torch.int32, device="cuda"), torch.zeros(4, dtype=torch.int32, device="cuda"),
                torch.zeros((2, 4), dtype=torch.int32, device="cuda")[:, ::2], good.tolist()):
        with pytest.raises(ValueError):
            dec.decode_crops_device(4, g, bad, (8, 8))
    with pytest.raises(hgi.HgiError):
        dec.decode_crops_device(4, g, good, (49, 8))
    torch.cuda.synchronize()
    ctx.close()
