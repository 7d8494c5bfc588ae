#!/usr/bin/env python
"""Scalable decode on one GPU: what a viewport, an overview or a batch of thumbnails costs against the full decode.

    python tools/bench_region.py [--calls 20] [--warmup 3]

Cases (one JSON line on stdout, with the card's name and power limit read in the same run):
  * config 4 (synthetic 16384^2, level 8, Medium), grid resident: full decode, a 1920x1080 viewport at (5000, 7000)
    (k = 0), overviews at k = 3 and k = 4;
  * 4096 x 1080p frames (level 4, Medium), grids resident: full decode, whole-batch thumbnails at k = 1 and k = 2;
  * host API: the viewport of a pinned 16384^2 grid (hgi_decode_region_u8) against hgi_decode_u8 of the whole plane.
Device cases are timed call by call with CUDA events, and 256 MB are written between calls so that every call starts
with an L2 that holds nothing of its inputs (a viewport's window would otherwise stay resident).  Host cases time the
synchronous call with a host clock.  The byte model counts DRAM bytes: the gather reads every 32-byte sector of the
window's grid rows the lattice touches (min(2^k, 32) bytes per point) and writes the dense window, the window decode
reads and writes the window, the crop reads and writes the region; a full decode reads and writes the plane.  Kernel
times of the gather and the crop come from torch.profiler in a separate pass; their GB/s are set against 6454.6 GB/s,
the copy bandwidth measured on a B200 (read + write bytes of a 2 GiB copy_) that the rooflines of profiles/ use."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np
import torch

import rustyhgi_b200 as hgi

COPY_PEAK_GBS = 6454.6


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = (s.strip() for s in out.split(","))
    except Exception as e:   # the number is still reported, without the power limit
        info["power_limit"] = f"unavailable ({e})"
    return info


def byte_model(w, h, n, k, region, levels):
    """DRAM bytes of one call: (gather, window decode, crop) for a region call, (0, 2 w h n, 0) for a full decode."""
    if k is None:
        return 0, 2 * w * h * n, 0
    pl = hgi.plan_region(w, h, levels, k, region)
    _, _, ww, wh = pl.window
    rw, rh = (pl.scaled_width, pl.scaled_height) if region is None else region[2:]
    gather = n * wh * (ww * min(1 << k, 32) + ((ww + 15) // 16) * 16)
    decode = 2 * n * ww * wh if pl.levels else 0
    crop = 2 * n * rw * rh
    return gather, decode, crop


def time_device(fn, calls, warmup, flush):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    total = 0.0
    for _ in range(calls):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
    return total / calls * 1e3


def kernel_us(fn, calls, flush):
    """Mean device time of the gather and crop kernels of `fn` (torch.profiler, CUDA activity)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            flush.fill_(1)
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for tag in ("gather", "crop"):
            if f"hgi_region_{tag}_kernel" in ev.key and ev.count:
                out[tag] = out.get(tag, 0.0) + ev.device_time_total / calls
    return out


def region_entry(name, w, h, n, k, region, levels, us, kern):
    g, d, c = byte_model(w, h, n, k, region, levels)
    e = {"case": name, "us_per_call": round(us, 2), "bytes": {"gather": g, "window_decode": d, "crop": c, "total": g + d + c},
         "bytes_per_full_res_pixel": round((g + d + c) / (w * h * n), 4)}
    for tag, b in (("gather", g), ("crop", c)):
        if tag in kern and kern[tag] > 0:
            gbs = b / (kern[tag] * 1e-6) / 1e9
            e[f"{tag}_kernel"] = {"us": round(kern[tag], 2), "GB_s": round(gbs, 1), "of_copy_peak": round(gbs / COPY_PEAK_GBS, 3)}
    return e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--frames", type=int, default=4096)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_region.py needs a CUDA device")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ctx = hgi.Context(0)
    dec = hgi.Decoder(hgi.Crossed, ctx=ctx)
    results = []

    # ---- config 4, grid resident
    n = 16384
    x = torch.arange(n, device="cuda", dtype=torch.int32)
    img = ((x[None, :] * x[:, None]) & 255).to(torch.uint8).contiguous()
    grid = hgi.Encoder(hgi.Crossed, hgi.Linear(hgi.QuantizationLevel.Medium), 8, ctx=ctx).encode_device(img)
    del img
    full = torch.empty_like(grid)
    us = time_device(lambda: dec.decode_device(8, grid, images_out=full), a.calls, a.warmup, flush)
    results.append(region_entry("c4 16384^2 L8: full decode", n, n, 1, None, None, 8, us, {}))
    for name, k, region in (("c4 viewport 1920x1080 at (5000,7000), k=0", 0, (5000, 7000, 1920, 1080)),
                            ("c4 overview k=3", 3, None), ("c4 overview k=4", 4, None)):
        pl = hgi.plan_region(n, n, 8, k, region)
        rw, rh = (pl.scaled_width, pl.scaled_height) if region is None else region[2:]
        out = torch.empty((rh, rw), dtype=torch.uint8, device="cuda")
        fn = lambda: dec.decode_region_device(8, grid, region=region, scale_log2=k, out=out)   # noqa: E731
        us = time_device(fn, a.calls, a.warmup, flush)
        s = full[::1 << k, ::1 << k]
        want = s if region is None else s[region[1]:region[1] + rh, region[0]:region[0] + rw]
        assert torch.equal(out, want), name
        results.append(region_entry(name, n, n, 1, k, region, 8, us, kernel_us(fn, 5, flush)))
    host_grid = grid.cpu().numpy()
    del grid, full

    # ---- 4096 x 1080p batch, grids resident
    fw, fh, nf = 1920, 1080, a.frames
    yy = torch.arange(fh, device="cuda", dtype=torch.int32)[:, None]
    xx = torch.arange(fw, device="cuda", dtype=torch.int32)[None, :]
    kk = torch.arange(nf, device="cuda", dtype=torch.int32)[:, None, None]
    frames = ((xx * yy + 31 * kk) & 255).to(torch.uint8).contiguous()
    grids = hgi.Encoder(hgi.Crossed, hgi.Linear(hgi.QuantizationLevel.Medium), 4, ctx=ctx).encode_device(frames)
    del frames
    full = torch.empty_like(grids)
    us = time_device(lambda: dec.decode_device(4, grids, images_out=full), a.calls, a.warmup, flush)
    results.append(region_entry(f"{nf} x 1080p L4: full decode", fw, fh, nf, None, None, 4, us, {}))
    for k in (1, 2):
        out = torch.empty((nf, -(-fh >> k), -(-fw >> k)), dtype=torch.uint8, device="cuda")
        fn = lambda: dec.decode_region_device(4, grids, scale_log2=k, out=out)   # noqa: E731
        us = time_device(fn, a.calls, a.warmup, flush)
        assert torch.equal(out, full[:, ::1 << k, ::1 << k]), k
        results.append(region_entry(f"{nf} x 1080p thumbnails k={k}", fw, fh, nf, k, None, 4, us, kernel_us(fn, 3, flush)))
        del out
    del grids, full

    # ---- host API, pinned 16384^2 grid
    L = hgi.lib()
    nb = n * n
    pg = L.hgi_host_alloc(nb)
    po = L.hgi_host_alloc(nb)
    assert pg and po, "hgi_host_alloc failed"
    g_np = np.ctypeslib.as_array((ctypes.c_uint8 * nb).from_address(pg))
    g_np[:] = host_grid.reshape(-1)
    p = hgi._lib.Params(8, 0, 0, 0)
    r = hgi._lib.RectStruct(5000, 7000, 1920, 1080)

    def host_time(call):
        for _ in range(a.warmup):
            ctx.check(call(), "host call")
        t0 = time.perf_counter()
        for _ in range(a.calls):
            ctx.check(call(), "host call")
        return (time.perf_counter() - t0) / a.calls * 1e6

    us_full = host_time(lambda: L.hgi_decode_u8(ctx._h, pg, n, n, ctypes.byref(p), po))
    us_view = host_time(lambda: L.hgi_decode_region_u8(ctx._h, pg, n, n, ctypes.byref(p), 0, ctypes.byref(r), po))
    view = np.ctypeslib.as_array((ctypes.c_uint8 * (1920 * 1080)).from_address(po)).reshape(1080, 1920).copy()
    ctx.check(L.hgi_decode_u8(ctx._h, pg, n, n, ctypes.byref(p), po), "hgi_decode_u8")
    whole = np.ctypeslib.as_array((ctypes.c_uint8 * nb).from_address(po)).reshape(n, n)
    assert np.array_equal(view, whole[7000:8080, 5000:6920])
    pl = hgi.plan_region(n, n, 8, 0, (5000, 7000, 1920, 1080))
    results.append({"case": "host API: hgi_decode_u8 16384^2 (pinned)", "us_per_call": round(us_full, 1),
                    "pcie_bytes": 2 * nb})
    results.append({"case": "host API: hgi_decode_region_u8 viewport 1920x1080 at (5000,7000) (pinned)",
                    "us_per_call": round(us_view, 1), "pcie_bytes": pl.window[2] * pl.window[3] + 1920 * 1080})
    L.hgi_host_free(pg)
    L.hgi_host_free(po)
    ctx.close()
    print(json.dumps({"tool": "bench_region", "gpu": card(), "calls": a.calls, "l2": "256 MB written between calls",
                      "copy_peak_GB_s": COPY_PEAK_GBS, "results": results}), flush=True)


if __name__ == "__main__":
    main()
