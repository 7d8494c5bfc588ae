#!/usr/bin/env python
"""Reduced parity subset for compute-sanitizer (one tool per gpurun call, B200_PROFILING.md):

    compute-sanitizer --tool memcheck|racecheck|initcheck python tools/sanitize_subset.py [--light]

Touches every kernel of libhgi_b200.so through the C ABI -- fast tile kernel (interior + edge launches, all level
counts, aligned / unaligned / pitched planes), decimated coarse passes,
histogram, RLE token table, RGB->luma, error metrics -- and checks each result against the oracle."""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch

import rustyhgi_b200 as hgi
from conftest import get_plane, photo_like
from oracle import c as oc

ap = argparse.ArgumentParser()
ap.add_argument("--light", action="store_true", help="smaller planes (racecheck is ~100x slower than memcheck)")
a = ap.parse_args()
Q = hgi.QuantizationLevel
n_checked = 0


def check(ctx, img, levels, q, interp=hgi.Crossed):
    global n_checked
    qi = oc.INTERP_CROSSED if interp is hgi.Crossed else oc.INTERP_LEFTTOP
    want_g, want_r = oc.encode(img, levels, interp=qi, qlevel=q, want_recon=True)
    enc = hgi.Encoder(interp, hgi.Linear(Q(q)), levels, ctx=ctx)
    grid, recon = enc.encode(img, want_recon=True)
    assert (grid.as_plane() == want_g).all() and (recon == want_r).all(), (img.shape, levels, q)
    assert (enc.encode(img).as_plane() == want_g).all()
    h, w = img.shape
    assert (hgi.Decoder(interp, ctx=ctx).decode((w, h), levels, grid) == want_r).all()
    n_checked += 1


paths = {"tile": hgi.PATH_TILE}
ctxs = {k: hgi.Context(0, v) for k, v in paths.items()}
lena = get_plane("lena_tif")
for name, ctx in ctxs.items():
    check(ctx, get_plane("unit_12x8"), 3, 2)
    check(ctx, lena, 4, 2)
    check(ctx, lena[:100, :131].copy(), 4, 1, interp=hgi.LeftTop)
    for (w, h, levels, q) in [(1, 1, 4, 2), (17, 9, 2, 3), (129, 65, 4, 0), (300, 70, 5, 2), (145, 81, 1, 1)]:
        check(ctx, photo_like(w, h, w + h), levels, q)
big = photo_like(640, 400, 5) if a.light else get_plane("fullhd")
check(ctxs["tile"], big, 4, 2)
check(ctxs["tile"], big, 4, 0)
check(ctxs["tile"], photo_like(700, 530, 6) if a.light else photo_like(2368, 1400, 6), 6, 3)      # decimated coarse pass
check(ctxs["tile"], photo_like(300, 1100, 9), 9, 2)                                                 # three passes

# interior + edge launches of the quantizing encode (>= 5920 tiles), batch API with histograms
ctx = ctxs["tile"]
n = 6 if a.light else 24
frames = np.stack([photo_like(1920, 1080, k) for k in range(n)]) if not a.light else np.stack([photo_like(1920, 1080, k) for k in range(n)])
if a.light:
    frames = frames[:, :400, :1024].copy()
    frames = np.concatenate([frames] * 8)               # 48 planes of 1024 x 400: 8 x 7 tiles each
want = oc.encode_batch(frames, 4, qlevel=2)
grids, hist = hgi.Encoder(hgi.Crossed, hgi.Linear(Q.Medium), 4, ctx=ctx).encode_batch(frames, want_hist=True)
assert (grids == want).all() and (hist[1] == np.bincount(want[1].reshape(-1), minlength=256)).all()
assert (hgi.Decoder(hgi.Crossed, ctx=ctx).decode_batch(4, grids) == oc.decode_batch(want, 4)).all()

# pitched planes and odd base addresses on the device API
for (w, h, levels, q, pad) in [(131, 65, 3, 1, 16), (1000, 120, 5, 2, 0), (37, 33, 6, 2, 32)]:
    pitch = (w + 15) // 16 * 16 + pad
    img = photo_like(w, h, w)
    wg, wr = oc.encode(img, levels, qlevel=q, want_recon=True)
    buf = torch.randint(0, 256, (1, h, pitch), dtype=torch.uint8, device="cuda")
    buf[0, :, :w] = torch.from_numpy(img).cuda()
    g = torch.zeros_like(buf)
    o = torch.zeros_like(buf)
    hh = torch.empty((1, 256), dtype=torch.int32, device="cuda")
    hgi.Encoder(hgi.Crossed, hgi.Linear(Q(q)), levels, ctx=ctx).encode_device(buf[:, :, :w], grids_out=g[:, :, :w], hist_out=hh)
    hgi.Decoder(hgi.Crossed, ctx=ctx).decode_device(levels, g[:, :, :w], images_out=o[:, :, :w])
    torch.cuda.synchronize()
    assert (g[0, :, :w].cpu().numpy() == wg).all() and (o[0, :, :w].cpu().numpy() == wr).all()
    assert (hh[0].cpu().numpy() == np.bincount(wg.reshape(-1), minlength=256)).all()
src = torch.zeros(70 * 131 + 64, dtype=torch.uint8, device="cuda")
img = photo_like(131, 70, 3)
src[3:3 + img.size] = torch.from_numpy(img).cuda().reshape(-1)
dst = torch.zeros_like(src)
hgi.Encoder(hgi.Crossed, hgi.Linear(Q.Low), 4, ctx=ctx).encode_device(src[3:3 + img.size].view(1, 70, 131), grids_out=dst[5:5 + img.size].view(1, 70, 131))
torch.cuda.synchronize()
assert (dst[5:5 + img.size].cpu().numpy().reshape(70, 131) == oc.encode(img, 4, qlevel=1)).all()

# reductions, RLE token table, colour conversion
from rle_model import rle_table
g = want[0]
assert (hgi.histogram(g, ctx=ctx) == np.bincount(g.reshape(-1), minlength=256)).all()
tab = np.zeros((1, 288), np.uint32)
ctx.check(hgi.lib().hgi_rle_histogram_u8(ctx._h, g.ctypes.data, g.size, g.size, 1, tab.ctypes.data), "rle")
assert (tab == rle_table(g)).all()
m = hgi.error_metrics(frames[0], oc.decode(want[0], 4), ctx=ctx)
assert m["max_abs"] <= 20
rgb = np.random.default_rng(1).integers(0, 256, (64, 80, 3)).astype(np.uint8)
assert (hgi.rgb_to_luma(rgb, ctx=ctx) == oc.rgb_to_luma(rgb)).all()
for c in ctxs.values():
    c.close()
print(f"sanitize subset ok: {n_checked} single-plane cases + batch + pitched + reductions, every result equal to the oracle")
