"""Planes taller than one launch grid holds (-m gpu): more than 65 535 lattice rows in a coarse pass's decimation, and
more than 65 535 tile rows (4 194 240 image rows) in a pass, which the launcher runs one image at a time in bands of
up to 65 535 tile rows.  Narrow planes keep each one small (16 x 8.4 M rows is 134 MB).  Every byte of grid,
reconstruction, histogram and decoded image is compared with the oracle, on the host API and on the device API (three
identical calls on one stream: plain, captured, replayed from the graph cache), and every call's kernel count with
tile_model.expected_launches.  Also: padded rows on a PATH_PER_LEVEL context, which runs the tile path like every
hgi_path_t value."""
import numpy as np
import pytest

import rustyhgi_b200 as hgi
from conftest import photo_like
from oracle import c as oc
from tile_model import expected_launches

pytestmark = pytest.mark.gpu
Q = hgi.QuantizationLevel

# (rows, width, row pitch of the device planes, images, levels, quantizer level, interpolator)
CASES = {
    "1048577x16-n2-L5": (1048577, 16, 16, 2, 5, Q.Medium, "crossed"),       # the L5 coarse pass decimates 65537 rows
    "1048577x17-L8": (1048577, 17, 17, 1, 8, Q.Medium, "crossed"),
    "4194305x16-n2-L4": (4194305, 16, 16, 2, 4, Q.Medium, "crossed"),       # 65537 tile rows: two bands per image
    "4194305x17-pitch32-L5": (4194305, 17, 32, 1, 5, Q.Medium, "crossed"),
    "4194305x16-L4-lossless-lefttop": (4194305, 16, 16, 1, 4, Q.Lossless, "lefttop"),
    "8388625x16-L8": (8388625, 16, 16, 1, 8, Q.Medium, "crossed"),          # 131073 tile rows: three bands
}
INTERPS = {"crossed": (hgi.Crossed, oc.INTERP_CROSSED), "lefttop": (hgi.LeftTop, oc.INTERP_LEFTTOP)}


def tall_plane(w, h, seed):
    """A slow wrapping ramp down the rows and across the columns, plus noise: every symbol, and fix-ups at 0 / 255."""
    rng = np.random.default_rng(seed)
    y = (np.arange(h, dtype=np.uint32) * 3 // 7).astype(np.uint8)
    x = (np.arange(w, dtype=np.uint32) * 11).astype(np.uint8)
    return y[:, None] + x[None, :] + rng.integers(0, 8, (h, w), dtype=np.uint8)   # uint8: wraps


def counted(ctx, fn):
    """(result of fn, kernels it launched, graphs it launched) on `ctx`."""
    k0, g0 = ctx.kernel_launches, ctx.graph_launches
    out = fn()
    return out, ctx.kernel_launches - k0, ctx.graph_launches - g0


@pytest.fixture(scope="module")
def ctx():
    c = hgi.Context(0)
    c.set_pipeline(4096, 0)    # a host call is one chunk: its kernel count is one device call's
    yield c
    c.close()


@pytest.mark.parametrize("case", list(CASES))
def test_tall_planes_equal_the_oracle(ctx, case):
    import torch
    h, w, pitch, n, levels, q, interp = CASES[case]
    cls, oid = INTERPS[interp]
    qerr = 10 * int(q)
    imgs = np.stack([tall_plane(w, h, 17 * k + h) for k in range(n)])
    want_g = oc.encode_batch(imgs, levels, interp=oid, qlevel=int(q))
    want_r = oc.decode_batch(want_g, levels, interp=oid)
    enc = hgi.Encoder(cls, hgi.Linear(q), levels, ctx=ctx)
    dec = hgi.Decoder(cls, ctx=ctx)

    # host API (packed rows)
    (grids, hist), k, _ = counted(ctx, lambda: enc.encode_batch(imgs, want_hist=True))
    assert np.array_equal(grids, want_g)
    for i in range(n):
        assert np.array_equal(hist[i], np.bincount(want_g[i].reshape(-1), minlength=256))
    assert k == expected_launches("enc", qerr, w, h, w % 16 == 0, levels, n, hist=True)
    if n == 1:
        (grid, recon), k, _ = counted(ctx, lambda: enc.encode(imgs[0], want_recon=True))
        assert np.array_equal(grid.as_plane(), want_g[0]) and np.array_equal(recon, want_r[0])
        assert k == expected_launches("enc", qerr, w, h, w % 16 == 0, levels, 1)
    back, k, _ = counted(ctx, lambda: dec.decode_batch(levels, want_g))
    assert np.array_equal(back, want_r)
    assert k == expected_launches("dec", 0, w, h, w % 16 == 0, levels, n)
    del grids, hist, back

    # device API, rows `pitch` bytes apart; the input's padding is garbage
    st = torch.cuda.Stream()
    src = torch.from_numpy(np.random.default_rng(h).integers(0, 256, (n, h, pitch), dtype=np.uint8)).cuda()
    src[:, :, :w] = torch.from_numpy(imgs).cuda()
    gbuf, rbuf, obuf = (torch.full((n, h, pitch), 0x5A, dtype=torch.uint8, device="cuda") for _ in range(3))
    dhist = torch.zeros((n, 256), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    graphs = (0, 1, 1) if levels > 4 else (0, 0, 0)     # chains of two passes or more are captured on their second call
    for rep in range(3):
        gbuf.fill_(0x5A), rbuf.fill_(0x5A), dhist.fill_(-1)
        torch.cuda.synchronize()
        _, k, g = counted(ctx, lambda: enc.encode_device(src[:, :, :w], grids_out=gbuf[:, :, :w], recon_out=rbuf[:, :, :w],
                                                         hist_out=dhist, stream=st.cuda_stream))
        st.synchronize()
        assert (k, g) == (expected_launches("enc", qerr, w, h, pitch % 16 == 0, levels, n, hist=True), graphs[rep]), rep
        assert np.array_equal(gbuf[:, :, :w].cpu().numpy(), want_g), rep
        assert np.array_equal(rbuf[:, :, :w].cpu().numpy(), want_r), rep
        for i in range(n):
            assert np.array_equal(dhist[i].cpu().numpy(), np.bincount(want_g[i].reshape(-1), minlength=256)), rep
    for rep in range(3):
        obuf.fill_(0x5A)
        torch.cuda.synchronize()
        _, k, g = counted(ctx, lambda: dec.decode_device(levels, gbuf[:, :, :w], images_out=obuf[:, :, :w], stream=st.cuda_stream))
        st.synchronize()
        assert (k, g) == (expected_launches("dec", 0, w, h, pitch % 16 == 0, levels, n), graphs[rep]), rep
        assert np.array_equal(obuf[:, :, :w].cpu().numpy(), want_r), rep


def test_pitched_planes_on_a_path_per_level_context():
    """PATH_PER_LEVEL runs the tile path, which takes padded rows (aligned and odd pitches) like HGI_PATH_TILE."""
    import torch
    c = hgi.Context(0, hgi.PATH_PER_LEVEL)
    for (n, h, w, pitch, levels, q) in [(2, 70, 131, 144, 4, 2), (1, 33, 37, 53, 6, 3), (2, 64, 40, 48, 3, 0)]:
        imgs = np.stack([photo_like(w, h, 5 * k + w) for k in range(n)])
        want_g = oc.encode_batch(imgs, levels, qlevel=q)
        want_r = oc.decode_batch(want_g, levels)
        src = torch.from_numpy(np.random.default_rng(w).integers(0, 256, (n, h, pitch), dtype=np.uint8)).cuda()
        src[:, :, :w] = torch.from_numpy(imgs).cuda()
        gbuf, rbuf, obuf = (torch.full((n, h, pitch), 0x5A, dtype=torch.uint8, device="cuda") for _ in range(3))
        hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels, ctx=c).encode_device(src[:, :, :w], grids_out=gbuf[:, :, :w],
                                                                                 recon_out=rbuf[:, :, :w])
        hgi.Decoder(hgi.Crossed, ctx=c).decode_device(levels, gbuf[:, :, :w], images_out=obuf[:, :, :w])
        torch.cuda.synchronize()
        tag = (n, h, w, pitch, levels, q)
        assert np.array_equal(gbuf[:, :, :w].cpu().numpy(), want_g), tag
        assert np.array_equal(rbuf[:, :, :w].cpu().numpy(), want_r), tag
        assert np.array_equal(obuf[:, :, :w].cpu().numpy(), want_r), tag
    c.close()
