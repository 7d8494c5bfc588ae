"""The pass/tile decomposition of the CUDA library, executed on the CPU (tests/tile_model.py),
must reproduce the oracle bit for bit -- including with every unstaged shared-memory byte
poisoned.  This checks the halo geometry (need_limit, staged rows, coarse fill) and the pass
plan without a GPU."""
import numpy as np
import pytest

import tile_model as tm
from conftest import photo_like
from oracle import c as oc


@pytest.mark.parametrize("w,h,levels,q", [(150, 70, 4, 2), (129, 65, 1, 3), (257, 129, 8, 3), (12, 8, 3, 2),
                                          (1, 1, 5, 2), (5, 1, 2, 1), (260, 70, 5, 2), (131, 67, 2, 1)])
def test_tile_model_matches_oracle(w, h, levels, q):
    img = photo_like(w, h, seed=w + 7 * h)
    table, _ = oc.quant_table(oc.QUANT_LINEAR, q)
    for crossed in (True, False):
        interp = oc.INTERP_CROSSED if crossed else oc.INTERP_LEFTTOP
        g, r = oc.encode(img, levels, interp=interp, qlevel=q, want_recon=True)
        g2, r2 = tm.encode(img, levels, table, crossed)
        assert (g == g2).all() and (r == r2).all()
        assert (tm.decode(g, levels, crossed) == r).all()


def test_small_tiles_many_passes():
    """Shrunken tiles (32x16) force many tiles and all three pass depths on a small plane."""
    img = photo_like(200, 90, 11)
    table, _ = oc.quant_table(oc.QUANT_LINEAR, 2)
    for levels in (1, 4, 6, 9):
        g, r = oc.encode(img, levels, qlevel=2, want_recon=True)
        g2, r2 = tm.encode(img, levels, table, True, tw=32, th=16)
        assert (g == g2).all() and (r == r2).all()
        assert (tm.decode(g, levels, True, tw=32, th=16) == r).all()


@pytest.mark.parametrize("args,kw,want", [
    (("enc", 20, 1920, 1080, True, 4, 4096), {"hist": True}, 4),   # the bench shape: interior + right column + bottom row + histogram
    (("enc", 20, 1920, 1080, True, 4, 23), {}, 1),                 # 23 * 255 tiles = 5865 < 5920: one launch
    (("enc", 20, 1920, 1080, True, 4, 24), {}, 3),                 # 24 * 255 = 6120 tiles split
    (("enc", 0, 1920, 1080, True, 4, 4096), {}, 1),                # Lossless never splits
    (("enc", 20, 1920, 1080, False, 4, 4096), {}, 1),              # nor the unaligned instantiation
    (("dec", 0, 1920, 1080, True, 4, 4096), {}, 1),
    (("enc", 20, 160, 96, True, 4, 1), {"split_min": 1}, 3),       # one interior tile, one right column (PART 2), one bottom row
    (("enc", 20, 256, 145, True, 4, 1), {"split_min": 1}, 3),      # 2 x 3 tiles, interior 1 x 2
    (("enc", 20, 128, 64, True, 4, 1), {"split_min": 1}, 1),       # no interior tile: the bottom-row launch only
    (("enc", 20, 160, 80, True, 4, 1), {"split_min": 1}, 1),       # an interior column but no interior row
    (("enc", 20, 96, 160, True, 4, 1), {"split_min": 1}, 1),       # an interior row but no interior column
    (("enc", 20, 160, 96, True, 5, 1), {"split_min": 1}, 5),       # decimate + coarse (1 level, one launch) + split fine pass
    (("enc", 20, 160, 96, True, 8, 1), {"split_min": 1, "hist": True}, 6),   # decimate + coarse split (bottom row only) + 3 + hist
    (("enc", 20, 2320, 1296, True, 8, 1), {"split_min": 1}, 7),    # the 145 x 81 coarse plane has an interior tile: 1 + 3 + 3
    (("dec", 0, 160, 96, True, 8, 1), {}, 3),
    (("enc", 20, 160, 96, True, 4, 66000), {"hist": True}, 5),     # 65535 images split, the remaining 465 (1860 tiles) do not
    (("enc", 20, 160, 96, True, 8, 66000), {}, 2 + 2 + 3 + 1),     # two decimate launches, two coarse chunks, split + plain fine
    (("enc", 20, 160, 96, True, 0, 3), {}, 0),                     # L = 0 is a copy
    (("enc", 20, 160, 96, True, 0, 3), {"hist": True}, 1),
    (("enc", 20, 0, 96, True, 4, 3), {"hist": True}, 0),
    # tall planes: the L5 coarse pass of 1048577 rows decimates 65537 lattice rows in two launches, 1025 tile rows
    (("dec", 0, 16, 1048577, True, 5, 1), {}, 2 + 1 + 1),
    # 65537 tile rows: per image a band of 65535 (no interior column: the bottom-row launch) and one of 2
    (("enc", 20, 16, 4194305, True, 4, 2), {"hist": True}, 2 * (1 + 1) + 1),
    (("enc", 20, 160, 4194305, True, 4, 1), {}, 2 + 1),           # band 0: interior + right column, band 1: 4 tiles, one launch
    # 131073 tile rows, three bands; the coarse pass decimates 524290 lattice rows in nine launches
    (("enc", 20, 16, 8388625, True, 8, 1), {}, 9 + 1 + 3),
    (("enc", 20, 160, 8388625, True, 4, 2), {}, 2 * (2 + 2 + 1)),
])
def test_expected_launches(args, kw, want):
    """The plain statement of the launch dispatch (tile_model.expected_launches) on hand-worked shapes."""
    assert tm.expected_launches(*args, **kw) == want


def test_pass_plan():
    assert tm.plan_passes(4) == [(0, 4)]
    assert tm.plan_passes(6) == [(4, 2), (0, 4)]
    assert tm.plan_passes(8) == [(4, 4), (0, 4)]
    assert tm.plan_passes(9) == [(8, 1), (4, 4), (0, 4)]
    assert tm.effective_levels(31, 1920, 1080) == 11
    assert tm.effective_levels(4, 1, 1) == 0
