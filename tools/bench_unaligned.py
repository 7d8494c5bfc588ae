#!/usr/bin/env python
"""Odd widths through the device API: packed planes (stride == width: 32-bit / funnel-shift / byte accesses when the
width is not a multiple of 16) against the same planes with rows padded to a 16-byte multiple (hgi_*_dev_pitched: the
128-bit path at any width).  256 planes of height 1080, Medium level 4; encode + decode Mpixel/s."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import rustyhgi_b200 as hgi


def t(fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


print("| width | layout | encode ms | decode ms | enc+dec Mpixel/s |\n|---|---|---|---|---|")
for w in (1920, 1916, 1918, 1919, 1000):
    pitch = (w + 15) // 16 * 16
    for layout in ("packed", "rows padded to %d" % pitch):
        if layout == "packed":
            frames = torch.randint(0, 256, (256, 1080, w), dtype=torch.uint8, device="cuda")
            g, o = torch.empty_like(frames), torch.empty_like(frames)
        else:
            if pitch == w:
                continue
            buf = torch.randint(0, 256, (256, 1080, pitch), dtype=torch.uint8, device="cuda")
            frames = buf[:, :, :w]
            g, o = torch.empty_like(buf)[:, :, :w], torch.empty_like(buf)[:, :, :w]
        ctx = hgi.Context(0)
        enc = hgi.Encoder(hgi.Crossed, hgi.Linear(hgi.QuantizationLevel.Medium), 4, ctx=ctx)
        dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
        te = t(lambda: enc.encode_device(frames, grids_out=g))
        td = t(lambda: dec.decode_device(4, g, images_out=o))
        print(f"| {w} | {layout} | {te:.3f} | {td:.3f} | {256 * 1080 * w / (te + td) / 1e3:.0f} |")
        ctx.close()
