"""Batched crops on the CPU: hgi_plan_crop against a plain statement of the uniform-window rule, its two promises (the
window's size does not depend on the origin, and the window contains hgi_plan_region's window of the same rectangle),
and the rule's claim -- decoding the planned window of the decimated grid with L' levels and cropping it equals slicing
the full decode -- checked with the oracle on seeded cases.  The GPU side is tests/test_gpu_crops.py."""
import ctypes

import numpy as np
import pytest

import rustyhgi_b200 as hgi
from conftest import photo_like
from oracle import c as oc


def axis(n, c, s, a, u):
    """DESIGN.md "Batched crops", one axis: (start, extent) of the window of a crop [u, u + c) of an n-cell axis."""
    need = c + 2 * s + a - 1
    d = n if need >= n else n - (n - need) // a * a
    return min(u // a * a, n - d), d


def plan(w, h, levels, k, crop):
    ws, hs = -(-w // (1 << k)), -(-h // (1 << k))
    x, y, cw, ch = crop
    lp = max(levels - k, 0)
    s = 1 << lp
    x0, dx = axis(ws, cw, s, max(s, 16), x)
    y0, dy = axis(hs, ch, s, s, y)
    return hgi.api.RegionPlan(ws, hs, lp, (x0, y0, dx, dy), x - x0, y - y0)


def random_shape(rng, max_side, max_levels, max_k=None):
    w, h = (int(v) for v in rng.integers(1, max_side + 1, 2))
    levels = int(rng.integers(0, max_levels + 1))
    k = int(rng.integers(0, (levels + 2) if max_k is None else max_k + 1))
    ws, hs = -(-w // (1 << k)), -(-h // (1 << k))
    return w, h, levels, k, ws, hs


def origins(rng, ws, hs, cw, ch, n_random=4):
    """Both corners, then random positions."""
    out = [(0, 0), (ws - cw, hs - ch), (0, hs - ch), (ws - cw, 0)]
    out += [(int(rng.integers(0, ws - cw + 1)), int(rng.integers(0, hs - ch + 1))) for _ in range(n_random)]
    return list(dict.fromkeys(out))


def test_plan_crop_matches_the_statement():
    rng = np.random.default_rng(11)
    cases = [(1920, 1080, 4, 0, (0, 0, 224, 224)), (1920, 1080, 4, 0, (1696, 856, 224, 224)),
             (16384, 16384, 8, 0, (5000, 7000, 1920, 1080)), (1, 1, 0, 0, (0, 0, 1, 1)), (1, 1, 31, 31, (0, 0, 1, 1)),
             (1919, 65, 12, 3, (7, 2, 1, 1)), (7, 5, 2, 5, (0, 0, 1, 1)), (2**26 - 1, 1, 31, 0, (2**25, 0, 3, 1))]
    for _ in range(500):
        w, h, levels, k, ws, hs = random_shape(rng, 5000, 13, 15)
        cw, ch = int(rng.integers(1, ws + 1)), int(rng.integers(1, hs + 1))
        x, y = int(rng.integers(0, ws - cw + 1)), int(rng.integers(0, hs - ch + 1))
        cases.append((w, h, levels, k, (x, y, cw, ch)))
    for w, h, levels, k, crop in cases:
        assert hgi.plan_crop(w, h, levels, k, crop) == plan(w, h, levels, k, crop), (w, h, levels, k, crop)
    # the worked example: a 224 x 224 crop of a 1080p L4 frame decodes a 272 x 280 window wherever it sits
    assert hgi.plan_crop(1920, 1080, 4, 0, (0, 0, 224, 224)).window == (0, 0, 272, 280)
    assert hgi.plan_crop(1920, 1080, 4, 0, (1696, 856, 224, 224)).window == (1648, 800, 272, 280)


def test_window_size_is_independent_of_the_origin_and_contains_the_region_window():
    rng = np.random.default_rng(12)
    for _ in range(400):
        w, h, levels, k, ws, hs = random_shape(rng, 3000, 12)
        cw, ch = int(rng.integers(1, ws + 1)), int(rng.integers(1, hs + 1))
        sizes = set()
        for x, y in origins(rng, ws, hs, cw, ch):
            pl = hgi.plan_crop(w, h, levels, k, (x, y, cw, ch))
            wx, wy, dx, dy = pl.window
            sizes.add((dx, dy))
            assert wx + dx <= ws and wy + dy <= hs
            s = 1 << pl.levels
            assert wx % max(s, 16) == 0 and wy % s == 0, (w, h, levels, k, pl)
            tx, ty, tw, th = hgi.plan_region(w, h, levels, k, (x, y, cw, ch)).window
            assert wx <= tx and wy <= ty and tx + tw <= wx + dx and ty + th <= wy + dy, (w, h, levels, k, (x, y, cw, ch))
            assert (pl.crop_x, pl.crop_y) == (x - wx, y - wy)
        assert len(sizes) == 1, (w, h, levels, k, cw, ch, sizes)


def crop_by_plan(grid, levels, k, crop, interp):
    h, w = grid.shape
    pl = plan(w, h, levels, k, crop)
    wx, wy, dx, dy = pl.window
    win = np.ascontiguousarray(grid[::1 << k, ::1 << k][wy:wy + dy, wx:wx + dx])
    dec = oc.decode(win, pl.levels, interp=interp)
    return dec[pl.crop_y:pl.crop_y + crop[3], pl.crop_x:pl.crop_x + crop[2]]


def crop_case(seed):
    """Sizes 1..300 (every 25th a 1-pixel plane), L 0..8, k 0..L+1 (k > L included), both interpolators, all four
    quantizer levels, random and photo-like planes; every 7th crop is the whole scaled image."""
    rng = np.random.default_rng(1000 + seed)
    w, h, levels, k, ws, hs = random_shape(rng, 300, 8)
    if seed % 25 == 0:
        w, h, ws, hs = 1, 1, 1, 1
    interp = (oc.INTERP_CROSSED, oc.INTERP_LEFTTOP)[seed % 2]
    qlevel = (seed // 2) % 4
    cw, ch = (ws, hs) if seed % 7 == 0 else (int(rng.integers(1, ws + 1)), int(rng.integers(1, hs + 1)))
    img = rng.integers(0, 256, (h, w)).astype(np.uint8) if seed % 3 == 0 else photo_like(w, h, seed)
    return rng, img, levels, k, interp, qlevel, cw, ch


@pytest.mark.parametrize("block", range(6))
def test_planned_window_decodes_to_the_slice(block):
    """300 seeded cases, each at both corners, the two other corners and four random origins."""
    for seed in range(50 * block, 50 * block + 50):
        rng, img, levels, k, interp, qlevel, cw, ch = crop_case(seed)
        grid = oc.encode(img, levels, interp=interp, qlevel=qlevel)
        full = oc.decode(grid, levels, interp=interp)[::1 << k, ::1 << k]
        hs, ws = full.shape
        for x, y in origins(rng, ws, hs, cw, ch):
            got = crop_by_plan(grid, levels, k, (x, y, cw, ch), interp)
            assert np.array_equal(got, full[y:y + ch, x:x + cw]), (seed, img.shape, levels, k, interp, qlevel, (x, y, cw, ch))


def test_plan_crop_rejects_invalid_arguments():
    L = hgi.lib()
    p = hgi._lib.RegionPlanStruct()

    def rc(w, h, levels, k, crop):
        r = ctypes.byref(hgi._lib.RectStruct(*crop)) if crop is not None else None
        return L.hgi_plan_crop(w, h, levels, k, r, ctypes.byref(p))

    assert rc(64, 48, 4, 0, (0, 0, 64, 48)) == 0
    assert rc(64, 48, 4, 2, (0, 0, 16, 12)) == 0
    assert rc(64, 48, 4, 2, (0, 0, 17, 12)) == -1          # wider than the 16 x 12 scaled image
    assert rc(64, 48, 4, 2, (15, 11, 1, 2)) == -1          # outside it
    assert rc(64, 48, 4, 2, (0, 0, 0, 5)) == -1            # empty
    assert rc(64, 48, 4, 2, (3, 3, 4, 0)) == -1
    assert rc(0, 48, 4, 0, (0, 0, 1, 1)) == -1             # the scaled image of an empty plane is empty
    assert rc(64, 48, 4, 32, (0, 0, 1, 1)) == -1           # scale_log2 > HGI_MAX_LEVELS
    assert rc(64, 48, 32, 0, (0, 0, 1, 1)) == -1
    assert rc(2**32 - 1, 1, 4, 0, (2**32 - 2, 0, 2**32 - 1, 1)) == -1   # x + width overflows 32 bits
    assert rc(64, 48, 4, 0, None) == -1                    # a crop is required
    assert L.hgi_plan_crop(64, 48, 4, 0, ctypes.byref(hgi._lib.RectStruct(0, 0, 1, 1)), None) == -1
    with pytest.raises(hgi.HgiError):
        hgi.plan_crop(64, 48, 4, 1, (30, 0, 3, 1))
    with pytest.raises(hgi.HgiError):
        hgi.plan_crop(64, 48, 4, 0, None)
    # the device entry point checks its arguments before touching a device
    prm = hgi._lib.Params(4, 0, 0, 0)
    buf = np.zeros(16, np.uint8)
    org = np.zeros(2, np.int32)
    assert L.hgi_decode_crops_dev(None, buf.ctypes.data, 1, 4, 4, 4, ctypes.byref(prm), 0, 2, 2, org.ctypes.data,
                                  buf.ctypes.data, 4, None) == -1
