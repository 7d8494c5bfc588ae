"""The reduction kernels of hgi_reduce_kernels.cu against plain references, on each of their code paths (-m gpu).

Every kernel there picks a path by pointer alignment, length and layout.  The host `_u8` entry points always hand it
a 256-byte-aligned slot buffer, so most cases here call the `_dev` entry points through ctypes on torch buffers, with
the data placed at chosen byte offsets:
- hgi_luma_kernel: the 128-bit path (RGB and luma bases 16-byte aligned: `vec_ok`) and the scalar `luma_of` path
  (any other base), every (r, g, b) triple; lengths 16k +- 1 put the vector body and the scalar tail in one launch.
- hgi_error_kernel: both bases aligned (`vec_ok`) or not, lengths 1 ... 17, around 16 blocks' worth and past the
  148 * 16-block grid, extreme contents, and 2^32 + 33 bytes of 0 against 255 (sums past any 32-bit partial).
- hgi_hist_kernel: packed batches whose images start at every misalignment (byte head, 128-bit body, byte tail),
  slices of 64 KiB ... 1 MiB, padded rows (the padding is not counted; blocks clamped to the rows), a bin at
  2^32 - 1, and hgi_histogram_u8 over more than 4 GiB in one pipeline chunk and in many.
- hgi_rle_hist_kernel: every run length 1 ... 1100 at segment phases up to 511, every RFC 1951 length symbol, block
  layouts up to 65 535 blocks; hgi_archive_serialize_rle accepts the tables and refuses a falsified one.
The references are plain: np.bincount in int64, sums in int64 or Python ints, oracle.c.rgb_to_luma and
tests/rle_model.rle_table.  The multi-GB device buffers are allocated once for the module."""
import ctypes
import io
import zlib

import numpy as np
import pytest

import rustyhgi_b200 as hgi
from oracle import c as oc
from rle_model import SYMS, len_sym, rle_table

pytestmark = pytest.mark.gpu

INVALID = -1
BIG = (1 << 32) + 33                   # bytes of the large error-metrics planes
GUARD = 0xA5                           # output bytes around a result, which no kernel may write


@pytest.fixture(scope="module")
def env():
    import torch
    ctx = hgi.Context(0)
    yield hgi.lib(), ctx, torch
    torch.cuda.synchronize()
    ctx.close()
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def big(env):
    """Two device planes of BIG + 1 bytes: all 0 and all 255."""
    L, ctx, torch = env
    zeros = torch.zeros(BIG + 1, dtype=torch.uint8, device="cuda")
    full = torch.full((BIG + 1,), 255, dtype=torch.uint8, device="cuda")
    yield zeros, full
    del zeros, full
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def cur_stream(torch):
    """The torch stream the buffers were written on (the C ABI reads NULL as the context's own stream, so the legacy
    default stream goes in as cudaStreamLegacy)."""
    return torch.cuda.current_stream().cuda_stream or 1


def at_offset(torch, src, off, pad=16):
    """A fresh device buffer holding `src` (host array or device tensor, 1-D uint8) at byte `off`; returns the buffer
    and the device address of the data.  torch's allocator returns 512-byte-aligned blocks, so `off` alone decides
    the alignment the kernel sees.  The caller holds the buffer until the kernel's result is read: once it is dropped
    the allocator hands its memory to the next tensor."""
    n = src.size if isinstance(src, np.ndarray) else src.numel()
    buf = torch.empty(n + off + pad, dtype=torch.uint8, device="cuda")
    assert buf.data_ptr() % 256 == 0
    buf[off:off + n].copy_(torch.from_numpy(src) if isinstance(src, np.ndarray) else src)
    return buf, buf.data_ptr() + off


def bincount_rows(data, n_images):
    """(n_images, 256) int64 counts of `n_images` equal consecutive slices of `data`."""
    n_per = data.size // n_images
    idx = (np.arange(data.size, dtype=np.int64) // n_per) * 256 + data
    return np.bincount(idx, minlength=n_images * 256).reshape(n_images, 256)


def mod3_counts(lo, hi):
    """{255 - r: #{i in [lo, hi) : i % 3 == r}} for arrays lo, hi (content 255 - (i mod 3))."""
    return {255 - r: (hi - r + 2) // 3 - (lo - r + 2) // 3 for r in range(3)}


# ---- RGB -> luma ---------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def triples(env):
    """All 2^24 (r, g, b) triples on the device and their luma by oracle.c (f32, no FMA, truncation)."""
    L, ctx, torch = env
    v = np.arange(1 << 24, dtype=np.uint32)
    rgb = np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], axis=1).astype(np.uint8).reshape(-1)
    want = oc.rgb_to_luma(rgb.reshape(1, -1, 3)).reshape(-1)
    return torch.from_numpy(rgb).cuda(), torch.from_numpy(want).cuda()


def luma_mismatches(env, d_rgb, d_want, rgb_off, out_off, stream=None):
    """hgi_rgb_to_luma_dev on d_rgb placed at byte rgb_off, luma written at byte out_off of a guarded buffer; returns
    (pixels that differ from d_want, guard bytes overwritten)."""
    L, ctx, torch = env
    n = d_want.numel()
    src_buf, src = at_offset(torch, d_rgb, rgb_off)
    out = torch.full((n + out_off + 16,), GUARD, dtype=torch.uint8, device="cuda")
    dst = out.data_ptr() + out_off
    ctx.check(L.hgi_rgb_to_luma_dev(ctx._h, src, n, dst, stream or cur_stream(torch)), "hgi_rgb_to_luma_dev")
    got = out[out_off:out_off + n]
    guards = torch.cat((out[:out_off], out[out_off + n:]))
    return int((got != d_want).sum()), int((guards != GUARD).sum())


@pytest.mark.parametrize("out_off", (0, 7))
@pytest.mark.parametrize("rgb_off", (0, 1, 3, 15))
def test_luma_every_triple_at_every_base_offset(env, triples, rgb_off, out_off):
    """Both bases 16-byte aligned: the PRMT / __fadd_rz vector path; any other offset: the scalar luma_of path.  Both
    must give the oracle's byte for every triple."""
    assert luma_mismatches(env, *triples, rgb_off, out_off) == (0, 0)


@pytest.mark.parametrize("n", (15, 17, 16 * 1000 - 1, 16 * 1000 + 1, (1 << 24) - 1, (1 << 25) + 1))
def test_luma_vector_body_and_scalar_tail_in_one_launch(env, triples, n):
    """16k +- 1 pixels on aligned bases: k groups of 16 on the vector path, the rest on luma_of in the same launch;
    2^25 + 1 pixels also make every thread walk the vector grid-stride loop more than once.  The same lengths on a
    misaligned base run luma_of throughout."""
    L, ctx, torch = env
    d_rgb, d_want = triples
    reps = -(-n // (1 << 24))
    rgb, want = d_rgb.repeat(reps)[:3 * n], d_want.repeat(reps)[:n]
    assert luma_mismatches(env, rgb, want, 0, 0) == (0, 0)
    assert luma_mismatches(env, rgb, want, 3, 0) == (0, 0)


def test_luma_on_a_side_stream(env, triples):
    """The kernel runs on the stream it is given: buffers written on a side stream, the call enqueued there."""
    L, ctx, torch = env
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        result = luma_mismatches(env, *triples, 0, 0, stream=side.cuda_stream)
    assert result == (0, 0)
    with torch.cuda.stream(side):
        result = luma_mismatches(env, *triples, 1, 7, stream=side.cuda_stream)
    assert result == (0, 0)


# ---- `hgi test` error metrics ----------------------------------------------------------------------------------------

ERR_LENGTHS = (1, 15, 16, 17, 16 * 256 * 64 - 1, 16 * 256 * 64 + 1,  # 16 blocks of 256 threads x 64 bytes, +- 1
               148 * 16 * 256 * 64 + 4099)                           # past the 148 * 16 blocks of the capped grid
ERR_OFFSETS = ((0, 0), (0, 9), (3, 0), (3, 9))                       # (before, after): only (0, 0) is `vec_ok`


def error_ref(a, b):
    d = a.astype(np.int64) - b.astype(np.int64)
    return int((d * d).sum()), int(np.abs(d).max())


def error_dev(env, d_before, d_after, n):
    L, ctx, torch = env
    out = torch.full((2,), -1, dtype=torch.int64, device="cuda")
    ctx.check(L.hgi_error_metrics_dev(ctx._h, d_before, d_after, n, out.data_ptr(), cur_stream(torch)),
              "hgi_error_metrics_dev")
    s, m = out.cpu().tolist()
    return s, m


@pytest.mark.parametrize("n", ERR_LENGTHS)
def test_error_metrics_dev_paths_and_contents(env, n):
    """Sum of squared differences and max |difference| of identical planes, 0 against 255 (65025 n, 255) both ways,
    one differing byte at the first, a middle and the last position, and noise -- on all four alignments."""
    L, ctx, torch = env
    rng = np.random.default_rng(n)
    a = rng.integers(0, 256, n, dtype=np.uint8)
    cases = {"identical": (a, a), "0 vs 255": (np.zeros(n, np.uint8), np.full(n, 255, np.uint8)),
             "255 vs 0": (np.full(n, 255, np.uint8), np.zeros(n, np.uint8)),
             "noise": (a, rng.integers(0, 256, n, dtype=np.uint8))}
    for where in sorted({0, n // 2, n - 1}):
        b = a.copy()
        b[where] ^= 0x80
        cases[f"byte {where}"] = (a, b)
    bad = {}
    for name, (a_, b_) in cases.items():
        want = error_ref(a_, b_)
        if name == "identical":
            assert want == (0, 0)
        if name.endswith("255") or name.startswith("255"):
            assert want == (65025 * n, 255)
        da, db = torch.from_numpy(a_).cuda(), torch.from_numpy(b_).cuda()
        for oa, ob in ERR_OFFSETS:
            (ba, pa), (bb, pb) = at_offset(torch, da, oa), at_offset(torch, db, ob)
            got = error_dev(env, pa, pb, n)
            if got != want:
                bad[(name, oa, ob)] = (got, want)
    assert not bad, bad


def test_error_metrics_dev_past_2_32_bytes(env, big):
    """2^32 + 33 bytes of 0 against 255: a sum of 65025 (2^32 + 33) that no 32-bit partial (per thread, warp or
    block) survives, on the vector path (aligned bases) and the scalar one (both bases + 1)."""
    zeros, full = big
    want = (65025 * BIG, 255)
    assert error_dev(env, zeros.data_ptr(), full.data_ptr(), BIG) == want
    assert error_dev(env, full.data_ptr() + 1, zeros.data_ptr() + 1, BIG) == want


def test_error_metrics_u8_in_chunks_and_whole(env):
    """hgi_error_metrics_u8 in 1 MiB pipeline chunks (four, the last ragged) and as one default chunk: the same sum,
    sd_int = sum // n and max as the reference."""
    L, ctx, torch = env
    rng = np.random.default_rng(11)
    n = 3 * (1 << 20) + 5
    a = rng.integers(0, 256, n, dtype=np.uint8)
    b = np.clip(a.astype(np.int16) + rng.integers(-20, 21, n), 0, 255).astype(np.uint8)
    b[n - 1] = 255 - a[n - 1] if a[n - 1] < 128 else 0                  # the largest difference in the last byte
    s, m = error_ref(a, b)
    try:
        for chunk_mb in (1, 0):
            ctx.set_pipeline(chunk_mb=chunk_mb)
            got = hgi.error_metrics(a, b, ctx=ctx)
            assert (got["sum_sq"], got["sd_int"], got["max_abs"]) == (s, s // n, m), chunk_mb
    finally:
        ctx.set_pipeline(0, 0)


# ---- residual histogram --------------------------------------------------------------------------------------------

HIST_SIZES = (1, 15, 16, 17, (64 << 10) - 1, (64 << 10) + 1, (1 << 20) - 1, (1 << 20) + 1, (5 << 20) + 7)


def hist_dev(env, ptr, n_per, n_images):
    L, ctx, torch = env
    out = torch.full((n_images, 256), -1, dtype=torch.int32, device="cuda")
    ctx.check(L.hgi_histogram_dev(ctx._h, ptr, n_per, n_images, out.data_ptr(), cur_stream(torch)), "hgi_histogram_dev")
    return out.cpu().numpy().view(np.uint32).astype(np.int64)


def hist_contents(total, rng):
    return {"noise": rng.integers(0, 256, total, dtype=np.uint8),
            "one symbol": np.full(total, 0x5A, np.uint8),
            # equal symbols in different lanes of a warp: the bin ^ 8 * lane row swizzle must keep them apart
            "255 - i mod 3": (255 - np.arange(total) % 3).astype(np.uint8)}


@pytest.mark.parametrize("n_images,n_per", [(k, s) for k in (1, 3) for s in HIST_SIZES] +
                         [(70000, s) for s in (1, 15, 16, 17)])
def test_histogram_dev_packed_batches(env, n_images, n_per):
    """n_images packed planes of n_per bytes at data offsets 0 and 5: an odd n_per starts every image at its own
    misalignment, so the byte head, the 128-bit body and the byte tail of each slice all occur; 5 Mi + 7 bytes cut into
    64 KiB slices.  Each image's 256 counts equal np.bincount of its bytes."""
    L, ctx, torch = env
    rng = np.random.default_rng(n_images * 1000003 + n_per)
    bad = {}
    for name, data in hist_contents(n_images * n_per, rng).items():
        want = bincount_rows(data, n_images)
        for off in (0, 5):
            buf, ptr = at_offset(torch, data, off)
            got = hist_dev(env, ptr, n_per, n_images)
            if not np.array_equal(got, want):
                rows = np.flatnonzero((got != want).any(axis=1))
                bad[(name, off)] = (len(rows), int(rows[0]))
    assert not bad, bad


@pytest.mark.parametrize("n_per", ((64 << 10) - 1, (64 << 10) + 1))
def test_histogram_dev_70000_images_with_bodies(env, n_per):
    """70 000 images of 64 Ki +- 1 bytes (4.6 GB): one block per image, every image at its own misalignment with a full
    128-bit body.  Contents made on the device; the reference counts follow from the index."""
    L, ctx, torch = env
    n_images = 70000
    total = n_images * n_per
    lo = np.arange(n_images, dtype=np.int64) * n_per
    for off in (0, 5):
        pattern = torch.tensor([255, 254, 253], dtype=torch.uint8, device="cuda").repeat(-(-total // 3))[:total]
        buf, ptr = at_offset(torch, pattern, off)
        del pattern
        want = np.zeros((n_images, 256), np.int64)
        for sym, cnt in mod3_counts(lo, lo + n_per).items():
            want[:, sym] = cnt
        assert np.array_equal(hist_dev(env, ptr, n_per, n_images), want), off
        buf[off:off + total].fill_(0x5A)
        want = np.zeros((n_images, 256), np.int64)
        want[:, 0x5A] = n_per
        assert np.array_equal(hist_dev(env, ptr, n_per, n_images), want), off
        del buf


@pytest.mark.parametrize("n", (592 * (64 << 10) + 3, 100_000_007, 700_000_001))
def test_histogram_dev_slice_sizes(env, n):
    """One large image: the launcher cuts it into slices of total / 592 rounded up to 16 KiB, clamped to
    [64 KiB, 1 MiB] -- 64 KiB, 176 KiB and 1 MiB here.  A noise block of 1 MiB + 13 bytes repeats, so the slices
    start at every phase of it."""
    L, ctx, torch = env
    rng = np.random.default_rng(n)
    blk = rng.integers(0, 256, (1 << 20) + 13, dtype=np.uint8)
    reps, rest = divmod(n, blk.size)
    want = np.bincount(blk, minlength=256).astype(np.int64) * reps + np.bincount(blk[:rest], minlength=256)
    data = torch.from_numpy(blk).cuda().repeat(reps + 1)[:n]
    for off in (0, 5):
        buf, ptr = at_offset(torch, data, off)
        assert np.array_equal(hist_dev(env, ptr, n, 1)[0], want), off
        del buf


def test_histogram_dev_bin_at_2_32_minus_1(env, big):
    """2^32 - 1 bytes of one symbol: that bin reads exactly 0xFFFFFFFF and every other bin 0, from an aligned base and
    from base + 1 (byte head and tail around 4096 slices of 1 MiB)."""
    zeros, full = big
    n = (1 << 32) - 1
    for buf, sym in ((full, 255), (zeros, 0)):
        for off in (0, 1):
            want = np.zeros((1, 256), np.int64)
            want[0, sym] = 0xFFFFFFFF
            assert np.array_equal(hist_dev(env, buf.data_ptr() + off, n, 1), want), (sym, off)


PAD = 200                                # row padding: a symbol no plane of the pitched test contains


def pitched_case(env, w, h, pitch, content, levels=0, n_images=3):
    """encode_device with hist_out on n_images planes of w x h in rows of `pitch` bytes.  The padding of the input
    and output rows holds PAD; levels 0 copies the image rows into the grid and leaves the grid's padding as it is,
    so a histogram that counted padding would show PAD.  Returns (got, want) (n_images, 256) counts."""
    L, ctx, torch = env
    imgs = torch.full((n_images, h, pitch), PAD, dtype=torch.uint8, device="cuda")
    imgs[:, :, :w] = torch.from_numpy(content.reshape(n_images, h, w)).cuda()
    grids = torch.full((n_images, h, pitch), PAD, dtype=torch.uint8, device="cuda")
    hist = torch.full((n_images, 256), -1, dtype=torch.int32, device="cuda")
    enc = hgi.Encoder(hgi.Crossed, hgi.NoOp(), levels, ctx=ctx)
    enc.encode_device(imgs[:, :, :w], grids_out=grids[:, :, :w], hist_out=hist)
    rows = grids[:, :, :w].cpu().numpy()
    if levels == 0:
        assert np.array_equal(rows, content.reshape(n_images, h, w))
    got = hist.cpu().numpy().view(np.uint32).astype(np.int64)
    return got, bincount_rows(rows.reshape(-1), n_images)


def test_histogram_pitched_rows_via_encode(env):
    """Padded rows (pitch w + 1, w + 15 and align16(w) + 16) of widths 1 ... 33 and heights 1, 2, 65: the histogram
    counts each row's w bytes, from each row's own alignment, and never the padding."""
    rng = np.random.default_rng(5)
    bad = {}
    for w in range(1, 34):
        for pitch in sorted({w + 1, w + 15, ((w + 15) & ~15) + 16}):
            for h in (1, 2, 65):
                total = 3 * w * h
                for name, content in (("noise", rng.integers(0, PAD, total, dtype=np.uint8)),
                                      ("one symbol", np.full(total, 0x5A, np.uint8)),
                                      ("255 - i mod 3", (255 - np.arange(total) % 3).astype(np.uint8))):
                    got, want = pitched_case(env, w, h, pitch, content)
                    if not np.array_equal(got, want):
                        bad[(w, pitch, h, name)] = int(got[:, PAD].sum())
    assert not bad, bad


@pytest.mark.parametrize("w,h", ((70001, 1), (70001, 2), (300007, 3), (100, 2000), (33, 65)))
def test_histogram_pitched_wide_rows(env, w, h):
    """Blocks of a padded plane own whole rows: with 70 001- and 300 007-byte rows the 64 KiB slices would give more
    blocks than rows, and the launcher clamps them to h; 100 x 2000 gives four blocks of 500 rows.  Also after an
    encode with levels (the grid then comes from the tile kernels)."""
    rng = np.random.default_rng(w * h)
    for levels in (0, 3):
        got, want = pitched_case(env, w, h, w + 15, rng.integers(0, PAD, 3 * w * h, dtype=np.uint8), levels)
        assert np.array_equal(got, want), levels


def test_histogram_u8_over_4_gib_in_one_chunk_and_many(env):
    """hgi_histogram_u8 over 2^32 + 4099 host bytes whose symbol 0 occurs more than 2^32 times, with pipeline chunks
    of 4096 MiB (cut to 4095 MiB: the device bins are 32-bit, and a 2^32-byte chunk once counted as empty), 4095 MiB
    and the default 1 GiB.  Nonzero patches straddle every chunk boundary; the reference is exact in int64."""
    L, ctx, torch = env
    n = (1 << 32) + 4099
    rng = np.random.default_rng(4)
    host = np.zeros(n, np.uint8)
    starts = [0, (1 << 30) - 8, (4095 << 20) - 8, (1 << 32) - 8, n - 16]
    want = np.zeros(256, np.int64)
    covered = 0
    for s in starts:
        patch = rng.integers(1, 256, 1000 if s == 0 else 16, dtype=np.uint8)
        host[s:s + patch.size] = patch
        want += np.bincount(patch, minlength=256)
        covered += patch.size
    want[0] += n - covered
    assert want[0] > 1 << 32
    own = hgi.Context(0)             # its 4 GiB slot buffers are freed with it
    try:
        for chunk_mb in (4096, 4095, 0):
            own.set_pipeline(chunk_mb=chunk_mb)
            got = hgi.histogram(host, ctx=own).astype(np.int64)
            assert np.array_equal(got, want), (chunk_mb, got[0], want[0])
    finally:
        own.close()


def test_batches_of_2_31_images_are_refused(env):
    """The histogram is one launch with a block or more per image, so a batch of 2^31 or more images is refused before
    any device work (its bins would take 2 TiB): hgi_histogram_dev and an encode with hist_out."""
    L, ctx, torch = env
    d = torch.zeros(1 << 12, dtype=torch.uint8, device="cuda")
    dh = torch.zeros(1 << 10, dtype=torch.int32, device="cuda")
    p = hgi._lib.Params(0, 0, 0, 0)
    before = ctx.kernel_launches
    for k in (1 << 31, 0xFFFFFFFF):
        assert L.hgi_histogram_dev(ctx._h, d.data_ptr(), 1, k, dh.data_ptr(), None) == INVALID, k
        assert L.hgi_histogram_dev(ctx._h, d.data_ptr(), 0, k, dh.data_ptr(), None) == INVALID, k
        assert L.hgi_encode_dev(ctx._h, d.data_ptr(), k, 1, 1, ctypes.byref(p), d.data_ptr(), None,
                                dh.data_ptr(), None) == INVALID, k
        assert L.hgi_encode_dev_pitched(ctx._h, d.data_ptr(), k, 1, 1, 16, ctypes.byref(p), d.data_ptr(),
                                        None, dh.data_ptr(), None) == INVALID, k
    assert ctx.kernel_launches == before
    ctx.synchronize()


# ---- run-length token tables ---------------------------------------------------------------------------------------

SEG = 512                                # HGI_RLE_SEGMENT_BYTES
# RFC 1951 3.2.5: literal/length code -> lengths it stands for
RFC1951_LENGTHS = ((257, 3, 3), (258, 4, 4), (259, 5, 5), (260, 6, 6), (261, 7, 7), (262, 8, 8), (263, 9, 9),
                   (264, 10, 10), (265, 11, 12), (266, 13, 14), (267, 15, 16), (268, 17, 18), (269, 19, 22),
                   (270, 23, 26), (271, 27, 30), (272, 31, 34), (273, 35, 42), (274, 43, 50), (275, 51, 58),
                   (276, 59, 66), (277, 67, 82), (278, 83, 98), (279, 99, 114), (280, 115, 130), (281, 131, 162),
                   (282, 163, 194), (283, 195, 226), (284, 227, 257), (285, 258, 258))
RFC_SYMBOL = {length: code for code, lo, hi in RFC1951_LENGTHS for length in range(lo, hi + 1)}


def rle_dev(env, data, block_bytes=None, off=0):
    """hgi_rle_histogram_dev of host `data` placed at byte `off`; (n_blocks, 288) int64."""
    L, ctx, torch = env
    n = data.size
    nb = 1 if block_bytes is None else -(-n // block_bytes)
    buf, ptr = at_offset(torch, data, off)
    out = torch.full((nb, SYMS), -1, dtype=torch.int32, device="cuda")
    ctx.check(L.hgi_rle_histogram_dev(ctx._h, ptr, n, block_bytes or n, nb, out.data_ptr(), cur_stream(torch)),
              "hgi_rle_histogram_dev")
    return out.cpu().numpy().view(np.uint32).astype(np.int64)


def rle_u8(env, data, block_bytes=None):
    L, ctx, torch = env
    nb = 1 if block_bytes is None else -(-data.size // block_bytes)
    out = np.zeros((nb, SYMS), np.uint32)
    ctx.check(L.hgi_rle_histogram_u8(ctx._h, data.ctypes.data, data.size, block_bytes or data.size, nb, out.ctypes.data),
              "hgi_rle_histogram_u8")
    return out.astype(np.int64)


def rle_archive(data, table, block_bytes=None):
    """hgi_archive_serialize_rle of `data` as a grid of width block_bytes (or data.size) with `table`; the raw
    DEFLATE payload."""
    width = block_bytes or data.size
    out = io.BytesIO()
    hgi.Archive(hgi.Metadata(0, 0, width, 1, 0), hgi.Grid(data, width)).serialize_to_writer(
        out, entropy="rle", hist=table, block_rows=1 if block_bytes else None)
    return out.getvalue()[28:]


def bincode_grid(data, width):
    return data.size.to_bytes(8, "little") + data.tobytes() + int(width).to_bytes(8, "little")


def phase_plane(phase, lengths=range(1, 1101)):
    """Runs of every length in `lengths`, each starting at byte `phase` of a 512-byte segment, so that a run crosses
    zero, one or two segment boundaries at that phase.  A filler run of another symbol pads to the next start; the
    run symbols step by 7 and so take all 256 values."""
    parts, pos, prev = [], 0, None
    for k, length in enumerate(lengths):
        v = (7 * k) % 256
        pad = (phase - pos) % SEG
        if pad:
            parts.append(np.full(pad, min(set(range(3)) - {prev, v}), np.uint8))
        parts.append(np.full(length, v, np.uint8))
        pos += pad + length
        prev = v
    return np.concatenate(parts)


def test_rle_every_run_length_at_every_segment_phase(env):
    """Runs of 1 ... 1100 bytes starting at offsets 0, 1, 254, 509, 510 and 511 of a segment: each side of a boundary
    is parsed on its own.  Device and host entry points equal rle_table; the union of the tables covers all 256
    literals and every length symbol 257 ... 285 (and never 286, 287), so a corpus that lost coverage fails here."""
    union = np.zeros(SYMS, np.int64)
    for phase in (0, 1, 254, 509, 510, 511):
        data = phase_plane(phase)
        want = rle_table(data).astype(np.int64)
        got = rle_dev(env, data)
        assert np.array_equal(got, want), (phase, np.flatnonzero(got != want)[:8])
        assert np.array_equal(rle_u8(env, data), want), phase
        union += got[0]
        if phase in (0, 509):              # the host writer accepts the device's tables
            assert zlib.decompress(rle_archive(data, got), -15) == bincode_grid(data, data.size)
    assert (union[:256] > 0).all(), np.flatnonzero(union[:256] == 0)
    assert (union[257:286] > 0).all(), 257 + np.flatnonzero(union[257:286] == 0)
    assert union[256] == 0 and (union[286:] == 0).all()


def test_rle_length_symbols_match_rfc1951(env):
    """The device rle_len_sym, symbol by symbol: block m - 3 of one plane holds a run of m + 1 bytes (one literal and
    one match of length m) and an alternating 1, 2 filler, so its table has exactly one length symbol, which must
    be the RFC 1951 code of m.  The host writer accepts these tables and refuses them once one count moves."""
    assert sorted(RFC_SYMBOL) == list(range(3, 259))
    assert all(len_sym(m) == RFC_SYMBOL[m] for m in range(3, 259))      # the CPU model states the same mapping
    blocks = []
    for m in range(3, 259):
        blk = np.resize(np.array([1, 2], np.uint8), SEG)
        blk[:m + 1] = 0
        blocks.append(blk)
    data = np.concatenate(blocks)
    got = rle_dev(env, data, SEG)
    assert np.array_equal(got, rle_table(data, SEG).astype(np.int64))
    bad = {}
    for b, m in enumerate(range(3, 259)):
        syms = 257 + np.flatnonzero(got[b, 257:])
        if list(syms) != [RFC_SYMBOL[m]] or got[b, RFC_SYMBOL[m]] != 1 or got[b, 0] != 1:
            bad[m] = list(syms)
    assert not bad, bad
    assert zlib.decompress(rle_archive(data, got, SEG), -15) == bincode_grid(data, SEG)
    moved = got.copy()
    b = 100                                 # match length 103: code 279
    moved[b, RFC_SYMBOL[103]] -= 1
    moved[b, RFC_SYMBOL[103] + 1] += 1
    with pytest.raises(hgi.HgiError) as e:
        rle_archive(data, moved, SEG)
    assert e.value.status == INVALID


def runs(rng, n, mean):
    """n bytes of runs of random symbols, lengths 1 ... 2 * mean."""
    lens = rng.integers(1, 2 * mean + 1, n // mean + 16)
    while lens.sum() < n:
        lens = np.concatenate((lens, rng.integers(1, 2 * mean + 1, n // mean + 16)))
    return np.repeat(rng.integers(0, 256, lens.size).astype(np.uint8), lens)[:n]


@pytest.mark.parametrize("n", (1, 2, 3, 511, 512, 513))
def test_rle_one_block(env, n):
    """n_blocks = 1 around one segment: a literal, a literal pair, the shortest match, a segment minus one, one
    segment, one segment and a byte."""
    rng = np.random.default_rng(n)
    for data in (np.full(n, 9, np.uint8), rng.integers(0, 256, n, dtype=np.uint8), runs(rng, n, 5)):
        want = rle_table(data).astype(np.int64)
        assert np.array_equal(rle_dev(env, data), want)
        assert np.array_equal(rle_dev(env, data, off=3), want)
        assert np.array_equal(rle_u8(env, data), want)
    assert zlib.decompress(rle_archive(data, rle_dev(env, data)), -15) == bincode_grid(data, n)


@pytest.mark.parametrize("block_bytes", (SEG, 7 * SEG))
@pytest.mark.parametrize("last", ("1 byte", "block - 1"))
def test_rle_many_blocks_with_a_short_last_one(env, block_bytes, last):
    """Five blocks of 512 or 3584 bytes, the last one 1 byte or block_bytes - 1 bytes long: each table describes its
    own block, segments counted from the block start; the archive of the device tables inflates to bincode(Grid)."""
    rng = np.random.default_rng(block_bytes)
    n = 4 * block_bytes + (1 if last == "1 byte" else block_bytes - 1)
    for data in (runs(rng, n, 40), runs(rng, n, 600)):
        want = rle_table(data, block_bytes).astype(np.int64)
        got = rle_dev(env, data, block_bytes)
        assert np.array_equal(got, want)
        assert np.array_equal(rle_dev(env, data, block_bytes, off=3), want)
        assert np.array_equal(rle_u8(env, data, block_bytes), want)
        assert zlib.decompress(rle_archive(data, got, block_bytes), -15) == bincode_grid(data, block_bytes)


def test_rle_65535_blocks_at_base_offset_3(env):
    """The largest grid the launcher takes: 65 535 blocks of 512 bytes (grid.y), the last one 100 bytes, data at
    base offset 3."""
    rng = np.random.default_rng(65535)
    n = 65534 * SEG + 100
    data = runs(rng, n, 60)
    want = rle_table(data, SEG).astype(np.int64)
    assert np.array_equal(rle_dev(env, data, SEG, off=3), want)
