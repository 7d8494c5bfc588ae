"""Scalable decode on the CPU: hgi_plan_region against a plain statement of the plan, and the plan's claim -- decoding
the planned window of the decimated grid with L' levels and cropping it equals slicing the full decode -- checked with
the oracle on seeded cases.  The GPU side is tests/test_gpu_region.py."""
import ctypes

import numpy as np
import pytest

import rustyhgi_b200 as hgi
from conftest import photo_like
from oracle import c as oc
from rustyhgi_b200 import cli


def plan(w, h, levels, k, region=None, end_cells=2):
    """The window rule of DESIGN.md "Scalable decode"; end_cells=1 is the shorter end bound that is not enough."""
    ws, hs = -(-w // (1 << k)), -(-h // (1 << k))
    x, y, rw, rh = region if region is not None else (0, 0, ws, hs)
    lp = max(levels - k, 0)
    s = 1 << lp
    a = max(s, 16)
    x0, y0 = x // a * a, y // s * s
    x1 = min(ws, (x + rw - 1) // s * s + end_cells * s + 1)
    y1 = min(hs, (y + rh - 1) // s * s + end_cells * s + 1)
    return hgi.api.RegionPlan(ws, hs, lp, (x0, y0, x1 - x0, y1 - y0), x - x0, y - y0)


def region_by_plan(grid, levels, k, region, interp, end_cells=2):
    h, w = grid.shape
    pl = plan(w, h, levels, k, region, end_cells)
    wx, wy, ww, wh = pl.window
    win = np.ascontiguousarray(grid[::1 << k, ::1 << k][wy:wy + wh, wx:wx + ww])
    dec = oc.decode(win, pl.levels, interp=interp)
    x, y, rw, rh = region
    return dec[pl.crop_y:pl.crop_y + rh, pl.crop_x:pl.crop_x + rw]


def random_case(seed):
    rng = np.random.default_rng(seed)
    w, h = (int(v) for v in rng.integers(1, 301, 2))
    levels = int(rng.integers(0, 9))
    k = int(rng.integers(0, levels + 2))
    interp = (oc.INTERP_CROSSED, oc.INTERP_LEFTTOP)[seed % 2]
    qlevel = (seed // 2) % 4
    ws, hs = -(-w // (1 << k)), -(-h // (1 << k))
    x, y = int(rng.integers(0, ws)), int(rng.integers(0, hs))
    region = (x, y, int(rng.integers(1, ws - x + 1)), int(rng.integers(1, hs - y + 1)))
    if seed % 3 == 0:
        img = rng.integers(0, 256, (h, w)).astype(np.uint8)
    else:
        img = photo_like(w, h, seed)
    return img, levels, k, interp, qlevel, region


def expected(img, levels, k, interp, qlevel, region):
    grid = oc.encode(img, levels, interp=interp, qlevel=qlevel)
    full = oc.decode(grid, levels, interp=interp)
    x, y, rw, rh = region
    return grid, full[::1 << k, ::1 << k][y:y + rh, x:x + rw]


def test_plan_region_matches_the_statement():
    rng = np.random.default_rng(7)
    cases = [(16384, 16384, 8, 0, (5000, 7000, 1920, 1080)), (16384, 16384, 8, 4, None), (16384, 16384, 8, 8, None),
             (1, 1, 0, 0, None), (1, 1, 31, 31, None), (1919, 65, 12, 3, (7, 2, 1, 1)), (7, 5, 2, 5, None)]
    for _ in range(500):
        w, h = (int(v) for v in rng.integers(1, 5000, 2))
        levels = int(rng.integers(0, 14))
        k = int(rng.integers(0, 16))
        ws, hs = -(-w // (1 << k)), -(-h // (1 << k))
        x, y = int(rng.integers(0, ws)), int(rng.integers(0, hs))
        cases.append((w, h, levels, k, (x, y, int(rng.integers(1, ws - x + 1)), int(rng.integers(1, hs - y + 1)))))
    for w, h, levels, k, region in cases:
        assert hgi.plan_region(w, h, levels, k, region) == plan(w, h, levels, k, region), (w, h, levels, k, region)
    # a 1920x1080 viewport of the 16384^2 level-8 plane reads a 2561 x 1537 window of the grid
    assert hgi.plan_region(16384, 16384, 8, 0, (5000, 7000, 1920, 1080)).window == (4864, 6912, 2561, 1537)


@pytest.mark.parametrize("block", range(6))
def test_planned_window_decodes_to_the_slice(block):
    """300 seeded cases (sizes 1..300, L 0..8, k 0..L+1, Crossed and LeftTop, all four quantizer levels, random and
    photo-like planes, random regions)."""
    for seed in range(50 * block, 50 * block + 50):
        img, levels, k, interp, qlevel, region = random_case(seed)
        grid, want = expected(img, levels, k, interp, qlevel, region)
        got = region_by_plan(grid, levels, k, region, interp)
        assert np.array_equal(got, want), (seed, img.shape, levels, k, interp, qlevel, region)


# (w, h, levels, k, interp, qlevel, region, seed): cases whose slice differs when the window ends one coarse cell
# earlier (end bound floor((u1 - 1) / S') * S' + S' + 1)
SHORT_BOUND_CASES = [
    (278, 58, 6, 1, oc.INTERP_CROSSED, 1, (2, 20, 5, 4), 49),
    (282, 124, 4, 0, oc.INTERP_CROSSED, 2, (132, 51, 94, 40), 94),
    (72, 231, 5, 3, oc.INTERP_CROSSED, 0, (7, 2, 2, 21), 68),
    (25, 233, 4, 1, oc.INTERP_CROSSED, 1, (11, 61, 1, 22), 0),
    (228, 267, 2, 0, oc.INTERP_CROSSED, 1, (99, 4, 36, 130), 55),
    (119, 296, 7, 0, oc.INTERP_CROSSED, 0, (33, 213, 18, 18), 99),
    (106, 102, 4, 0, oc.INTERP_CROSSED, 1, (88, 51, 9, 26), 24),
    (63, 221, 5, 1, oc.INTERP_CROSSED, 2, (15, 0, 16, 42), 0),
]


def test_end_bound_needs_two_coarse_cells():
    short_differs = 0
    for w, h, levels, k, interp, qlevel, region, seed in SHORT_BOUND_CASES:
        img = photo_like(w, h, seed)
        grid, want = expected(img, levels, k, interp, qlevel, region)
        assert np.array_equal(region_by_plan(grid, levels, k, region, interp), want)
        short_differs += not np.array_equal(region_by_plan(grid, levels, k, region, interp, end_cells=1), want)
    assert short_differs == len(SHORT_BOUND_CASES)


def test_plan_region_rejects_invalid_arguments():
    L = hgi.lib()
    p = hgi._lib.RegionPlanStruct()

    def rc(w, h, levels, k, region):
        r = ctypes.byref(hgi._lib.RectStruct(*region)) if region is not None else None
        return L.hgi_plan_region(w, h, levels, k, r, ctypes.byref(p))

    assert rc(64, 48, 4, 0, None) == 0
    assert rc(64, 48, 4, 2, (0, 0, 16, 12)) == 0
    assert rc(64, 48, 4, 2, (0, 0, 17, 12)) == -1          # outside the 16 x 12 scaled image
    assert rc(64, 48, 4, 2, (15, 11, 1, 2)) == -1
    assert rc(64, 48, 4, 2, (0, 0, 0, 5)) == -1            # empty
    assert rc(64, 48, 4, 2, (3, 3, 4, 0)) == -1
    assert rc(0, 48, 4, 0, None) == -1                     # the scaled image of an empty plane is empty
    assert rc(64, 48, 4, 32, None) == -1                   # scale_log2 > HGI_MAX_LEVELS
    assert rc(64, 48, 32, 0, None) == -1
    assert rc(2**32 - 1, 1, 4, 0, (2**32 - 2, 0, 2**32 - 1, 1)) == -1   # x + width overflows 32 bits
    assert L.hgi_plan_region(64, 48, 4, 0, None, None) == -1
    with pytest.raises(hgi.HgiError):
        hgi.plan_region(64, 48, 4, 1, (30, 0, 3, 1))
    # the device entry points check their arguments before touching a device
    prm = hgi._lib.Params(4, 0, 0, 0)
    buf = np.zeros(16, np.uint8)
    assert L.hgi_decode_region_u8(None, buf.ctypes.data, 4, 4, ctypes.byref(prm), 0, None, buf.ctypes.data) == -1
    assert L.hgi_decode_region_dev(None, buf.ctypes.data, 1, 4, 4, 4, ctypes.byref(prm), 0, None, buf.ctypes.data, 4, None) == -1


def test_cli_parses_scale_and_region():
    a = cli.build_parser().parse_args(["decode", "-i", "x.hgi", "-o", "y.png", "--scale", "2", "--region", "5,6,70,80"])
    assert a.scale == 2 and a.region == (5, 6, 70, 80)
    a = cli.build_parser().parse_args(["decode", "-i", "x.hgi", "-o", "y.png"])
    assert a.scale == 0 and a.region is None
    for bad in (["--region", "1,2,3"], ["--region", "a,b,c,d"], ["--region", "1,2,-3,4"], ["--scale", "-1"]):
        with pytest.raises(SystemExit):
            cli.build_parser().parse_args(["decode", "-i", "x.hgi", "-o", "y.png"] + bad)
