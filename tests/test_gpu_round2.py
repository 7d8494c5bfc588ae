"""Round-2 additions to the GPU parity suite (-m gpu; all through the C ABI): planes with padded rows
(hgi_*_dev_pitched), coarse passes through the decimated dense plane, per-stream scratch (multi-chunk host batches with
levels > 4 and concurrent device-API streams on one context), size limits."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import rustyhgi_b200 as hgi
from conftest import photo_like
from oracle import c as oc

pytestmark = pytest.mark.gpu
Q = hgi.QuantizationLevel
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ctx():
    c = hgi.Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("path", [hgi.PATH_TILE, hgi.PATH_TILE_GENERIC])
def test_pitched_planes_any_width(path):
    """Rows padded to a 16-byte multiple (and further, and to odd pitches that take the unaligned instantiation): the
    padding bytes of the input are garbage and must not influence anything; grid, reconstruction, decoded image and histogram equal the oracle on the packed plane."""
    import torch
    c = hgi.Context(0, path)
    rng = np.random.default_rng(5)
    cases = [(2, 70, 1919, 4, 2, 0), (1, 65, 131, 3, 1, 16), (2, 129, 255, 5, 3, 0), (1, 33, 37, 6, 2, 32),
             (1, 300, 1000, 9, 2, 0), (3, 64, 128, 4, 0, 48), (1, 17, 1, 2, 1, 0), (1, 200, 145, 4, 2, 0),
             (2, 70, 131, 4, 2, 5), (1, 90, 256, 5, 3, 3), (2, 40, 64, 3, 1, 1)]      # pitches that are not multiples of 16 (or 4)
    for (n, h, w, levels, q, extra) in cases:
        pitch = (w + 15) // 16 * 16 + extra
        imgs = np.stack([photo_like(w, h, 3 * k + w) for k in range(n)])
        want_g = oc.encode_batch(imgs, levels, qlevel=q)
        want_r = oc.decode_batch(want_g, levels)
        buf = torch.from_numpy(rng.integers(0, 256, (n, h, pitch)).astype(np.uint8)).cuda()
        buf[:, :, :w] = torch.from_numpy(imgs).cuda()
        src = buf[:, :, :w]
        gbuf = torch.full((n, h, pitch), 0x5A, dtype=torch.uint8, device="cuda")
        rbuf = torch.full((n, h, pitch), 0x5A, dtype=torch.uint8, device="cuda")
        obuf = torch.full((n, h, pitch), 0x5A, dtype=torch.uint8, device="cuda")
        hist = torch.empty((n, 256), dtype=torch.int32, device="cuda")
        enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels, ctx=c)
        enc.encode_device(src, grids_out=gbuf[:, :, :w], recon_out=rbuf[:, :, :w], hist_out=hist)
        hgi.Decoder(hgi.Crossed, ctx=c).decode_device(levels, gbuf[:, :, :w], images_out=obuf[:, :, :w])
        torch.cuda.synchronize()
        tag = (n, h, w, levels, q, pitch)
        assert (gbuf[:, :, :w].cpu().numpy() == want_g).all(), tag
        assert (rbuf[:, :, :w].cpu().numpy() == want_r).all() and (obuf[:, :, :w].cpu().numpy() == want_r).all(), tag
        for k in range(n):
            assert (hist[k].cpu().numpy() == np.bincount(want_g[k].reshape(-1), minlength=256)).all(), tag
    c.close()


def test_deep_hierarchies_take_the_decimated_coarse_passes(ctx):
    """levels 5..12 on planes large enough for two and three passes: the coarse passes run on the gathered lattice."""
    rng = np.random.default_rng(8)
    for (w, h, levels, q) in [(2368, 1300, 6, 3), (1030, 2070, 8, 2), (4100, 530, 9, 1), (600, 5000, 12, 2), (4097, 4097, 12, 0)]:
        img = photo_like(w, h, levels) if q else rng.integers(0, 256, (h, w)).astype(np.uint8)
        want_g, want_r = oc.encode(img, levels, qlevel=q, want_recon=True)
        grid, recon = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels, ctx=ctx).encode(img, want_recon=True)
        assert (grid.as_plane() == want_g).all() and (recon == want_r).all(), (w, h, levels, q)
        assert (hgi.Decoder(hgi.Crossed, ctx=ctx).decode((w, h), levels, grid) == want_r).all()


_CHUNK_SCRIPT = r"""
import sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {root!r} + "/tests")
import numpy as np
import rustyhgi_b200 as hgi
from conftest import photo_like
from oracle import c as oc
for path in (hgi.PATH_TILE, hgi.PATH_PER_LEVEL):
    ctx = hgi.Context(0, path)
    for levels in (5, 6, 9):
        n, h, w = 14, 520, 650                      # 338 KB per plane: 3 planes per 1 MB chunk, 5 chunks over 3 slots
        imgs = np.stack([photo_like(w, h, 11 * k + levels) for k in range(n)])
        want_g = oc.encode_batch(imgs, levels, qlevel=2)
        want_r = oc.decode_batch(want_g, levels)
        for rep in range(3):
            grids, hist = hgi.Encoder(hgi.Crossed, hgi.Linear(hgi.QuantizationLevel.Medium), levels, ctx=ctx).encode_batch(imgs, want_hist=True)
            back = hgi.Decoder(hgi.Crossed, ctx=ctx).decode_batch(levels, grids)
            assert (grids == want_g).all() and (back == want_r).all(), (path, levels, rep)
            assert (hist[5] == np.bincount(want_g[5].reshape(-1), minlength=256)).all()
    ctx.close()
print("chunks ok")
"""


def test_multi_chunk_batches_keep_their_coarse_planes_apart():
    """ADVICE r1: chunks in flight on different slot streams used to share one set of compact coarse planes.  With
    1 MB chunks a 14-plane batch is five chunks on three streams; levels 5, 6, 9 need the coarse planes."""
    env = dict(os.environ, HGI_B200_CHUNK_MB="1")
    r = subprocess.run([sys.executable, "-c", _CHUNK_SCRIPT.format(root=ROOT)], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "chunks ok" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]


def test_concurrent_streams_on_one_context(ctx):
    """Device API on several caller streams of one context at once (levels > 4: every stream needs scratch planes)."""
    import torch
    levels, q, n_streams = 6, 2, 4
    imgs = [photo_like(1500, 900, 40 + k) for k in range(n_streams)]
    want = [oc.encode(im, levels, qlevel=q, want_recon=True) for im in imgs]
    streams = [torch.cuda.Stream() for _ in range(n_streams)]
    src = [torch.from_numpy(im).cuda() for im in imgs]
    grids = [torch.empty_like(s) for s in src]
    outs = [torch.empty_like(s) for s in src]
    torch.cuda.synchronize()
    enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels, ctx=ctx)
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    for rep in range(20):
        for k, st in enumerate(streams):
            enc.encode_device(src[k], grids_out=grids[k], stream=st.cuda_stream)
        for k, st in enumerate(streams):
            dec.decode_device(levels, grids[k], images_out=outs[k], stream=st.cuda_stream)
    torch.cuda.synchronize()
    for k in range(n_streams):
        assert (grids[k].cpu().numpy() == want[k][0]).all() and (outs[k].cpu().numpy() == want[k][1]).all(), k


def test_row_length_limit(ctx):
    L = hgi.lib()
    p = hgi._lib.Params(3, 0, 1, 2)
    one = np.zeros(16, np.uint8)
    assert L.hgi_encode_dev(ctx._h, one.ctypes.data, 1, 1 << 26, 1, ctypes.byref(p), one.ctypes.data, None, None, None) == -1
    assert L.hgi_decode_dev_pitched(ctx._h, one.ctypes.data, 1, 16, 1, 8, ctypes.byref(p), one.ctypes.data, None) == -1   # pitch < width


def _pool_devices():
    """All visible GPUs; on a single-GPU box two contexts on device 0 (the pool logic is the same)."""
    import torch
    n = torch.cuda.device_count()
    return list(range(n)) if n > 1 else [0, 0]


def test_pool_batch_by_image_equals_the_oracle():
    """hgi_pool_*_batch_u8: contiguous image shares on every member (SURVEY.md 8e row 1), with per-image histograms."""
    pool = hgi.Pool(_pool_devices())
    assert len(pool) >= 2
    n, h, w, levels, q = 4 * len(pool) + 3, 270, 480, 4, 2
    imgs = np.stack([photo_like(w, h, 5 * k + 1) for k in range(n)])
    want_g = oc.encode_batch(imgs, levels, qlevel=q)
    want_r = oc.decode_batch(want_g, levels)
    enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels)
    grids, hist = pool.encode_batch(enc, imgs, want_hist=True)
    back = pool.decode_batch(hgi.Decoder(hgi.Crossed), levels, grids)
    assert (grids == want_g).all() and (back == want_r).all()
    for k in (0, n // 2, n - 1):
        assert (hist[k] == np.bincount(want_g[k].reshape(-1), minlength=256)).all()
    one = pool.encode_batch(enc, imgs[:1])            # fewer images than members: the empty shares are skipped
    assert (one == want_g[:1]).all()
    pool.close()


def test_pool_row_bands_equal_the_full_plane():
    """hgi_pool_*_plane_u8 and the device-resident band calls: bands of multiples of S rows plus S + 1 overlap rows,
    no exchange (SURVEY.md 8e row 2; dependency direction: src/interpolator.rs:67-73)."""
    import torch
    pool = hgi.Pool(_pool_devices())
    for (w, h, levels, q) in [(1024, 2048 + 77, 8, 2), (640, 1000, 5, 1), (333, 517, 4, 3), (256, 100, 8, 2)]:
        img = photo_like(w, h, levels + w)
        want_g, want_r = oc.encode(img, levels, qlevel=q, want_recon=True)
        enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels)
        dec = hgi.Decoder(hgi.Crossed)
        grid = pool.encode_plane(enc, img)
        assert (grid.as_plane() == want_g).all(), (w, h, levels)
        assert (pool.decode_plane(dec, (w, h), levels, grid) == want_r).all(), (w, h, levels)
        # device-resident bands, called three times with the same buffers: the second call captures the launch chain
        # of every member, the third replays it
        bands = pool.plan_bands(h, levels)
        assert bands[0][0] == 0 and bands[-1][1] == h and all(b[0] % (1 << levels) == 0 for b in bands)
        devs = pool.devices
        d_in = [torch.from_numpy(img[y0:iy1]).to(f"cuda:{devs[k]}") for k, (y0, y1, iy1) in enumerate(bands)]
        d_grid = [torch.empty_like(t) for t in d_in]
        d_gin = [torch.from_numpy(want_g[y0:iy1]).to(f"cuda:{devs[k]}") for k, (y0, y1, iy1) in enumerate(bands)]
        d_out = [torch.empty_like(t) for t in d_in]
        for rep in range(3):
            pool.encode_bands_device(enc, d_in, w, h, d_grid)
            pool.decode_bands_device(dec, levels, d_gin, w, h, d_out)
            pool.synchronize()
            for k, (y0, y1, iy1) in enumerate(bands):
                assert (d_grid[k][:y1 - y0].cpu().numpy() == want_g[y0:y1]).all(), (w, h, levels, k, rep)
                assert (d_out[k][:y1 - y0].cpu().numpy() == want_r[y0:y1]).all(), (w, h, levels, k, rep)
    pool.close()


def test_launch_chains_are_replayed_from_graphs(ctx):
    """Identical device-API calls with three or more launches (levels > 4) are captured on the second call and
    replayed afterwards; results stay bit-exact and the kernel count keeps counting."""
    import torch
    w, h, levels, q = 2000, 1100, 7, 2
    img = photo_like(w, h, 99)
    want_g, want_r = oc.encode(img, levels, qlevel=q, want_recon=True)
    t = torch.from_numpy(img).cuda()
    g = torch.empty_like(t)
    o = torch.empty_like(t)
    st = torch.cuda.Stream()
    enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels, ctx=ctx)
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    torch.cuda.synchronize()
    g0, l0 = ctx.graph_launches, ctx.kernel_launches
    per_call = None
    for rep in range(5):
        before = ctx.kernel_launches
        enc.encode_device(t, grids_out=g, stream=st.cuda_stream)
        if per_call is None:
            per_call = ctx.kernel_launches - before
        assert ctx.kernel_launches - before == per_call
        dec.decode_device(levels, g, images_out=o, stream=st.cuda_stream)
        st.synchronize()
        assert (g.cpu().numpy() == want_g).all() and (o.cpu().numpy() == want_r).all(), rep
    assert per_call >= 3
    assert ctx.graph_launches - g0 == 2 * 4          # calls 2..5 of encode and of decode
    # another buffer: a different chain, plain launches again, still exact
    g2 = torch.empty_like(t)
    enc.encode_device(t, grids_out=g2, stream=st.cuda_stream)
    st.synchronize()
    assert (g2.cpu().numpy() == want_g).all()


def test_whole_tile_right_column_bodies(ctx):
    """Planes whose width is a multiple of the tile width (128) have exactly one non-interior tile column: decode and the
    identity encode run it through a body with constant extents (EDGE = 2) inside the kernel, the quantizing encode as a
    launch of its own when the job is large.  Heights around the tile-row and halo boundaries (64 k + 0..17), one to
    three interior tile rows, noise (every fix-up path) and a photograph-like plane."""
    rng = np.random.default_rng(21)
    for w in (128, 256, 640):
        for h in (64, 81, 82, 128 + 17, 128 + 18, 200, 3 * 64 + 1):
            for q in (0, 2):
                imgs = np.stack([rng.integers(0, 256, (h, w)).astype(np.uint8), photo_like(w, h, w + h)])
                want_g = oc.encode_batch(imgs, 4, qlevel=q)
                want_r = oc.decode_batch(want_g, 4)
                enc = hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), 4, ctx=ctx)
                grids = enc.encode_batch(imgs)
                assert (grids == want_g).all(), (w, h, q)
                assert (hgi.Decoder(hgi.Crossed, ctx=ctx).decode_batch(4, grids) == want_r).all(), (w, h, q)
