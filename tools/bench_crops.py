#!/usr/bin/env python
"""Batched crops on one GPU: a same-sized crop at its own random origin from every grid of a resident batch, against
the two ways a caller had before.

    python tools/bench_crops.py [--calls 20] [--warmup 3] [--frames 1024]

Setup: `--frames` resident 1080p grids (level 4, Medium).  Every call first draws new origins on the device
(torch.randint), as a training pipeline's random crop does, so no call reuses the last one's origins.  Cases: 224 x 224
crops at k = 0, 256 x 256 at k = 1, 128 x 128 at k = 2, each timed three ways:
  * crops:       one Decoder.decode_crops_device call (hgi_decode_crops_dev);
  * full+gather: Decoder.decode_device of the whole batch, then a torch gather of the crops out of the decoded frames;
  * region loop: the origins copied to the host, then one Decoder.decode_region_device call per plane.
Each call is timed with CUDA events; 256 MB are written between calls (outside the timed window) so that every call
starts with an L2 that holds nothing of its inputs.  The median of `--calls` calls is reported, after `--warmup` calls.
The byte model counts DRAM bytes per crop: the gather reads every 32-byte sector of the window's grid rows the lattice
touches (min(2^k, 32) bytes per point) and writes the dense window, the window decode reads and writes it, the crop
reads and writes the rectangle; a full decode reads and writes the frame, and its torch gather reads and writes the
crop.  The card's name and power limit are read in the same run.  One JSON line on stdout."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import rustyhgi_b200 as hgi

W, H, LEVELS = 1920, 1080, 4
CASES = ((0, 224), (1, 256), (2, 128))   # (scale_log2, crop side)


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = (s.strip() for s in out.split(","))
    except Exception as e:   # the number is still reported, without the power limit
        info["power_limit"] = f"unavailable ({e})"
    return info


def window_bytes(k, window, levels, cw, ch):
    """(gather, window decode, crop) DRAM bytes of one plane decoded from `window` (x, y, width, height)."""
    _, _, ww, wh = window
    gather = wh * (ww * min(1 << k, 32) + ((ww + 15) // 16) * 16)
    return gather, (2 * ww * wh if levels else 0), 2 * cw * ch


def time_device(fn, calls, warmup, flush):
    """Median milliseconds of `fn` over `calls` calls (CUDA events), with L2 overwritten before each."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(calls):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), float(min(ms)), float(max(ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", type=int, default=1024)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_crops.py needs a CUDA device")
    if a.calls < 20:
        sys.exit("--calls must be at least 20")
    gpu = card()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ctx = hgi.Context(0)
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    n = a.frames
    yy = torch.arange(H, device="cuda", dtype=torch.int32)[:, None]
    xx = torch.arange(W, device="cuda", dtype=torch.int32)[None, :]
    kk = torch.arange(n, device="cuda", dtype=torch.int32)[:, None, None]
    frames = ((xx * yy + 31 * kk) & 255).to(torch.uint8).contiguous()
    grids = hgi.Encoder(hgi.Crossed, hgi.Linear(hgi.QuantizationLevel.Medium), LEVELS, ctx=ctx).encode_device(frames)
    del frames
    full = torch.empty_like(grids)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(0)
    results = []
    for k, side in CASES:
        ws, hs = -(-W >> k), -(-H >> k)
        origins = torch.empty((n, 2), dtype=torch.int32, device="cuda")
        out = torch.empty((n, side, side), dtype=torch.uint8, device="cuda")
        ar = torch.arange(side, device="cuda")
        idx = torch.arange(n, device="cuda")[:, None, None]

        def draw():
            origins[:, 0] = torch.randint(0, ws - side + 1, (n,), device="cuda", dtype=torch.int32, generator=gen)
            origins[:, 1] = torch.randint(0, hs - side + 1, (n,), device="cuda", dtype=torch.int32, generator=gen)

        def crops():
            draw()
            dec.decode_crops_device(LEVELS, grids, origins, (side, side), scale_log2=k, out=out)

        def full_gather():
            draw()
            dec.decode_device(LEVELS, grids, images_out=full)
            s = full[:, ::1 << k, ::1 << k]
            rows = (origins[:, 1].long()[:, None] + ar)[:, :, None]
            cols = (origins[:, 0].long()[:, None] + ar)[:, None, :]
            out.copy_(s[idx, rows, cols])

        def region_loop():
            draw()
            xy = origins.cpu().tolist()   # the host must see every origin before it can plan
            for i, (x, y) in enumerate(xy):
                dec.decode_region_device(LEVELS, grids[i], region=(x, y, side, side), scale_log2=k, out=out[i])

        # every way gives the same bytes for the same origins
        draw()
        xy = origins.clone()
        dec.decode_crops_device(LEVELS, grids, xy, (side, side), scale_log2=k, out=out)
        got = out.clone()
        dec.decode_device(LEVELS, grids, images_out=full)
        s = full[:, ::1 << k, ::1 << k]
        want = s[idx, (xy[:, 1].long()[:, None] + ar)[:, :, None], (xy[:, 0].long()[:, None] + ar)[:, None, :]]
        assert torch.equal(got, want), (k, side)
        for i in (0, n // 2, n - 1):
            x, y = xy[i].tolist()
            assert torch.equal(dec.decode_region_device(LEVELS, grids[i], region=(x, y, side, side), scale_log2=k), want[i])

        pl = hgi.plan_crop(W, H, LEVELS, k, (0, 0, side, side))
        g, d, c = window_bytes(k, pl.window, pl.levels, side, side)
        tight = hgi.plan_region(W, H, LEVELS, k, (ws // 2 - side // 2, hs // 2 - side // 2, side, side))
        tg, td, tc = window_bytes(k, tight.window, tight.levels, side, side)
        per_crop = {"crops": g + d + c, "full+gather": 2 * W * H + 2 * side * side, "region loop": tg + td + tc}
        entry = {"case": f"{side}x{side} crops at k={k}", "window": list(pl.window[2:]), "levels_on_window": pl.levels,
                 "bytes_per_crop": {"gather": g, "window_decode": d, "crop": c}, "ways": {}}
        for name, fn in (("crops", crops), ("full+gather", full_gather), ("region loop", region_loop)):
            med, lo, hi = time_device(fn, a.calls, a.warmup, flush)
            entry["ways"][name] = {"ms_median": round(med, 3), "ms_min": round(lo, 3), "ms_max": round(hi, 3),
                                   "bytes_per_crop_model": per_crop[name],
                                   "GB_s_model": round(per_crop[name] * n / (med * 1e-3) / 1e9, 1)}
        results.append(entry)
        del out, origins
    ctx.close()
    print(json.dumps({"tool": "bench_crops", "gpu": gpu, "frames": n, "levels": LEVELS, "calls": a.calls,
                      "warmup": a.warmup, "statistic": "median of calls, CUDA events",
                      "l2": "256 MB written between calls", "results": results}), flush=True)


if __name__ == "__main__":
    main()
