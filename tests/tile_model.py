"""Executable model of the fused tile-pass decomposition used by the CUDA library
(the tile kernel of rustyhgi_b200/csrc/hgi_tile_fast.cu + plan_passes in hgi_capi.cu), stated byte by byte.

Test infrastructure: it mirrors, tile by tile, *which* bytes a CTA stages, which coarse values it
takes from the previous pass, which cells/points it processes per level (the `need_limit`
geometry) and what it writes back -- with every unstaged shared-memory byte poisoned -- so the
halo-sufficiency argument of DESIGN.md can be checked against the oracle on the CPU.
"""
import numpy as np

TW, TH, FMAX = 128, 64, 16
RPITCH, RROWS = TW + 32, TH + FMAX + 1
MAX_PASS_LEVELS = 4


def effective_levels(levels, w, h):
    m = max(w, h)
    need = 0
    while (1 << need) < m:
        need += 1
    return min(levels, need)


def plan_passes(levels):
    out, d, rem = [], 0, levels
    while rem > 0:
        nl = min(rem, MAX_PASS_LEVELS)
        out.append((d, nl))
        d += nl
        rem -= nl
    return out[::-1]


SPLIT_MIN_TILES = 4 * 1480      # split_min_tiles() in hgi_tile_fast.cu (HGI_B200_SPLIT_MIN overrides it)
MAX_GRID = 65535                 # images (gridDim.z) and rows (gridDim.y) per launch


def expected_launches(mode, qerr, w, h, pitch_aligned, levels, n, split_min=SPLIT_MIN_TILES, hist=False):
    """Kernels one device-API call of the tile path launches (hgi_ctx_kernel_launches), stated plainly: per pass of
    plan_passes(L), for a coarse pass one decimate launch per 65535 images x 65535 lattice rows; then per slice -- up to
    65535 whole images, or, in a plane of more than 65535 tile rows, one image's band of up to 65535 tile rows -- either
    one launch or, for a split quantizing encode, the interior / right-column / bottom-row launches that have tiles;
    plus one for the histogram.  `mode` is "enc" or "dec", `qerr` the quantizer's error (0: Lossless / NoOp),
    `pitch_aligned` whether the fine pass runs the 128-bit instantiation (16-byte rows and bases; coarse passes always
    do)."""
    if n == 0 or w * h == 0:
        return 0
    total = 1 if hist else 0
    chunks = [min(MAX_GRID, n - first) for first in range(0, n, MAX_GRID)]
    for (d, nlev) in plan_passes(effective_levels(levels, w, h)):
        wD, hD = -(-w >> d), -(-h >> d)
        tx, ty = -(-wD // TW), -(-hD // TH)
        if d > 0:
            total += len(chunks) * -(-hD // MAX_GRID)
        if ty <= MAX_GRID:   # (images, tile rows, rows from the slice's first row to the bottom of the plane)
            slices = [(cnt, ty, hD) for cnt in chunks]
        else:
            slices = [(1, min(MAX_GRID, ty - t0), hD - t0 * TH) for _ in range(n) for t0 in range(0, ty, MAX_GRID)]
        for cnt, rows, hr in slices:
            split = mode == "enc" and qerr != 0 and (pitch_aligned or d > 0) and nlev == 4 and tx * rows * cnt >= split_min
            if not split:
                total += 1
                continue
            itx = min(tx, (wD - (FMAX + 1)) // TW) if wD >= FMAX + 1 else 0
            ity = min(rows, (hr - (FMAX + 1)) // TH) if hr >= FMAX + 1 else 0
            if itx == 0 or ity == 0:
                itx = ity = 0
            total += (itx > 0) + (tx - itx > 0 and ity > 0) + (rows - ity > 0)
    return total


def need_limit(extent, s):
    return extent - 1 if s == 1 else (extent if s == 2 else extent + s)


def staged_rows():
    return list(range(TH)) + [TH, TH + 4, TH + 8]


def _predict(A, B, C, D, crossed):
    if not crossed:
        return A
    return (((A + B + 1) >> 1) + ((D + C + 1) >> 1) + ((C + A + 1) >> 1) + ((D + B + 1) >> 1)) >> 2


def run_pass(mode, src, d_log2, nlev, c_recon, c_q, table, crossed, rng, tw=TW, th=TH):
    """One pass over one plane.  Returns (q_lattice, recon_lattice) as wD x hD arrays."""
    h, w = src.shape
    D = 1 << d_log2
    lat = src[::D, ::D]
    hD, wD = lat.shape
    F = 1 << nlev
    top = c_recon is None
    out_q = np.zeros((hD, wD), np.uint8)
    out_r = np.zeros((hD, wD), np.uint8)
    for Y0 in range(0, hD, th):
        for X0 in range(0, wD, tw):
            xin = min(tw + FMAX + 1, wD - X0)
            yin = min(th + FMAX + 1, hD - Y0)
            R = rng.integers(0, 256, (th + FMAX + 1, tw + 32)).astype(np.int64)   # poison
            Q = rng.integers(0, 256, (th, tw)).astype(np.int64)
            rows = list(range(th)) + [th, th + 4, th + 8]
            for r in rows:                                    # staging
                for x in range(tw + 16):
                    R[r, x] = lat[Y0 + r, X0 + x] if (r < yin and x < xin) else 0
            for cj in range(th // F + 2):                     # coarse fill
                for ci in range(tw // F + 2):
                    x, y = ci * F, cj * F
                    rv = qv = 0
                    if x < xin and y < yin:
                        if top:
                            rv = qv = int(lat[Y0 + y, X0 + x])
                        else:
                            rv = int(c_recon[(Y0 + y) >> nlev, (X0 + x) >> nlev])
                            if mode == "enc":
                                qv = int(c_q[(Y0 + y) >> nlev, (X0 + x) >> nlev])
                    R[y, x] = rv
                    if x < tw and y < th:
                        Q[y, x] = qv
            s = F >> 1
            while s >= 1:
                step = 2 * s
                xlim, ylim = need_limit(tw, s), need_limit(th, s)
                ncx = tw // step + (1 if s >= 2 else 0)
                ncy = th // step + (1 if s >= 2 else 0)
                writes = []
                for cy in range(ncy):
                    for cx in range(ncx):
                        x0, y0 = cx * step, cy * step
                        if x0 >= xin or y0 >= yin:
                            continue
                        p = _predict(R[y0, x0], R[y0 + step, x0], R[y0, x0 + step], R[y0 + step, x0 + step], crossed)
                        for (x, y) in ((x0 + s, y0), (x0, y0 + s), (x0 + s, y0 + s)):
                            if x > xlim or y > ylim or x >= xin or y >= yin:
                                continue
                            if mode == "enc":
                                a = R[y, x]
                                d = (a - p) & 255
                                q = int(table[d])
                                if ((p + q) > 255) != ((p + d) > 255):
                                    q = d
                                if x < tw and y < th:
                                    Q[y, x] = q
                                writes.append((y, x, (p + q) & 255))
                            else:
                                writes.append((y, x, (p + R[y, x]) & 255))
                for (y, x, v) in writes:                      # a level only reads the coarser lattice
                    R[y, x] = v
                s >>= 1
            xo, yo = min(tw, xin), min(th, yin)
            out_r[Y0:Y0 + yo, X0:X0 + xo] = R[:yo, :xo]
            out_q[Y0:Y0 + yo, X0:X0 + xo] = Q[:yo, :xo]
    return out_q, out_r


def encode(image, levels, table, crossed=True, seed=0, tw=TW, th=TH):
    image = np.asarray(image, np.uint8)
    h, w = image.shape
    L = effective_levels(levels, w, h)
    if L == 0:
        return image.copy(), image.copy()
    rng = np.random.default_rng(seed)
    c_recon = c_q = None
    for (d, nl) in plan_passes(L):
        c_q, c_recon = run_pass("enc", image, d, nl, c_recon, c_q, table, crossed, rng, tw, th)
    return c_q, c_recon


def decode(grid, levels, crossed=True, seed=0, tw=TW, th=TH):
    grid = np.asarray(grid, np.uint8)
    h, w = grid.shape
    L = effective_levels(levels, w, h)
    if L == 0:
        return grid.copy()
    rng = np.random.default_rng(seed)
    c_recon = None
    for (d, nl) in plan_passes(L):
        _, c_recon = run_pass("dec", grid, d, nl, c_recon, None, None, crossed, rng, tw, th)
    return c_recon
