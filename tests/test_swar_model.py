"""Bit-level model of the 16-bit-lane SWAR arithmetic in rustyhgi_b200/csrc/hgi_tile_fast.cu,
checked exhaustively against the reference formulas (CPU only).  The device code uses exactly
these word operations; the GPU parity tests check the code, this checks the algebra."""
import itertools

import numpy as np

from oracle import c as oc

M16 = 0x00FF00FF
U32 = 0xFFFFFFFF


def ref_pred(A, B, C, D):
    avg = lambda x, y: (x + y + 1) >> 1                      # src/interpolator.rs:44
    return (avg(A, B) + avg(D, C) + avg(C, A) + avg(D, B)) >> 2


def swar_pred(A, B, C, D):                                    # pred2<Crossed> of round 1 (integer shift form)
    x1 = (A ^ B) & 0x00010001
    w = x1 & (C ^ D) & (A ^ C)
    t1 = (A + B + C) + (D + 0x00010001)                       # T + 1 per lane
    return ((t1 + 2 * w) >> 2) & M16                          # == (((T + 1) >> 1) + w) >> 1


def test_parity_predictor_all_low_bit_patterns_and_ranges():
    vals = [0, 1, 2, 3, 4, 5, 126, 127, 128, 129, 252, 253, 254, 255]
    for A, B, C, D in itertools.product(vals, repeat=4):
        assert swar_pred(A, B, C, D) == ref_pred(A, B, C, D)
    rng = np.random.default_rng(0)
    q = rng.integers(0, 256, (200000, 8))
    for A, B, C, D, A2, B2, C2, D2 in q[:20000]:
        lanes = swar_pred(int(A | (A2 << 16)), int(B | (B2 << 16)), int(C | (C2 << 16)), int(D | (D2 << 16)))
        assert lanes & 0xFFFF == ref_pred(A, B, C, D) and lanes >> 16 == ref_pred(A2, B2, C2, D2)


QUANT = {10: (195, 195, 12), 20: (25, 0, 10), 30: (67, 67, 12)}   # quant_swar()


def swar_encode2(a, p, error):
    """encode2<false> of round 1 (integer multiply-shift quantizer): returns (q lanes, recon lanes)."""
    k, c, n = QUANT[error]
    scale = 2 * error + 1
    add = ((error * k + c) * 0x00010001) & U32
    pk = (0x01000100 - p) & U32
    dd = (a + pk) & U32
    d = dd & M16
    t = (d * k + add) & U32
    rmask = ((0xF << n) * 0x00010001) & U32
    q = ((t & rmask) * (scale << (32 - n))) >> 32             # __umulhi
    ov = (q + p) & U32
    x = (~(ov ^ dd)) & 0x01000100
    m = min(x & 0xFFFF, 0xFF) | (min(x >> 16, 0xFF) << 16)     # min.u16x2(x, 0x00FF00FF): 0x00FF per mismatching lane
    q = (q & ~m & U32) | (dd & m)                             # dd's flag bit lies outside m
    recon = (a + q - d) & U32                                 # no borrow between lanes once the fix-up ran
    return q, recon


def ref_encode(a, p, table):
    d = (a - p) & 255                                          # src/encoder.rs:53
    q = int(table[d])                                          # :54
    if ((p + q) > 255) != ((p + d) > 255):                     # :56-58
        q = d
    return q, (p + q) & 255


def test_swar_encode_point_exhaustive():
    """All (a, p) pairs in both lanes, every Linear level: symbol and reconstruction."""
    for level, error in ((1, 10), (2, 20), (3, 30)):
        table, _ = oc.quant_table(oc.QUANT_LINEAR, level)
        for p0 in range(256):
            p1 = 255 - p0
            for a0 in range(256):
                a1 = (a0 * 7 + 13) & 255
                q, r = swar_encode2(a0 | (a1 << 16), p0 | (p1 << 16), error)
                q0, r0 = ref_encode(a0, p0, table)
                q1, r1 = ref_encode(a1, p1, table)
                assert (q & 0xFFFF, r & 0xFFFF, q >> 16, r >> 16) == (q0, r0, q1, r1), (level, a0, p0)


def test_swar_quantizer_constants_are_exact():
    for error, (k, c, n) in QUANT.items():
        scale = 2 * error + 1
        for d in range(256):
            t = d * k + error * k + c
            assert t < 65536 and ((t >> n) & 15) * scale == ((d + error) // scale) * scale
            assert ((t & (0xF << n)) * (scale << (32 - n))) >> 32 == ((d + error) // scale) * scale


def test_pack_lo_drops_the_carry_bits():
    """pack_lo (PRMT 0x6240) keeps only the low byte of every lane, so wrapping adds need no mask."""
    rng = np.random.default_rng(1)
    for _ in range(2000):
        p0, p1, g0, g1, h0, h1 = (int(v) for v in rng.integers(0, 256, 6))
        even = (p0 + g0) | ((p1 + g1) << 16)                   # 9-bit sums in both lanes
        odd = (p0 + h0) | ((p1 + h1) << 16)
        b = [even & 255, odd & 255, (even >> 16) & 255, (odd >> 16) & 255]
        packed = b[0] | (b[1] << 8) | (b[2] << 16) | (b[3] << 24)
        # __byte_perm(even, odd, 0x6240): result byte i = source byte selector nibble i (0-3 even, 4-7 odd)
        src = [(even >> (8 * i)) & 255 for i in range(4)] + [(odd >> (8 * i)) & 255 for i in range(4)]
        sel = 0x6240
        got = sum(src[(sel >> (4 * i)) & 7] << (8 * i) for i in range(4))
        assert got == packed
        assert [got & 255, (got >> 16) & 255] == [(p0 + g0) & 255, (p1 + g1) & 255]


def test_dirty_predictor_lanes_are_harmless_for_decode():
    """Round 1's decode skipped the shift-form predictor's final mask: the lanes then carry stray bits 14/15 (lane 1's low bits after the >> 2), which
    must never reach a low byte nor carry into the other lane when a clean residual lane is added."""
    rng = np.random.default_rng(7)
    for _ in range(20000):
        v = [int(x) for x in rng.integers(0, 256, 12)]
        A, B, C, D = (v[i] | (v[i + 4] << 16) for i in range(4))
        x1 = (A ^ B) & 0x00010001
        w = x1 & (C ^ D) & (A ^ C)
        t1 = (A + B + C) + (D + 0x00010001)
        p_dirty = (t1 + 2 * w) >> 2
        p_clean = p_dirty & M16
        g = v[8] | (v[9] << 16)
        r_d, r_c = (p_dirty + g) & U32, (p_clean + g) & U32
        assert r_d < (1 << 32) and (r_d & 0x00FF00FF) == (r_c & 0x00FF00FF)


def byte_perm(a, b, sel):
    src = [(a >> (8 * i)) & 255 for i in range(4)] + [(b >> (8 * i)) & 255 for i in range(4)]
    return sum(src[(sel >> (4 * i)) & 7] << (8 * i) for i in range(4))


def test_pack_even_row_selectors():
    """pack_even_row: bytes [c0, q0, c1, q1] from two consecutive bytes of the coarser symbol word and the low bytes
    of the two 16-bit lanes of the new symbols (clean lanes, or dirty ones for the identity quantizer)."""
    rng = np.random.default_rng(3)
    for _ in range(2000):
        qw = int(rng.integers(0, 1 << 32))
        q0, q1, junk0, junk1 = (int(v) for v in rng.integers(0, 256, 4))
        for lanes in (q0 | (q1 << 16), q0 | (junk0 << 8) | (q1 << 16) | (junk1 << 24)):
            lo = byte_perm(qw, lanes, 0x6140)
            hi = byte_perm(qw, lanes, 0x6342)
            assert lo == (qw & 255) | (q0 << 8) | (((qw >> 8) & 255) << 16) | (q1 << 24)
            assert hi == ((qw >> 16) & 255) | (q0 << 8) | (((qw >> 24) & 255) << 16) | (q1 << 24)


def test_lanewise_bias_tolerates_dirty_predictor_lanes():
    """Round 1's bias_sub: pk = ~p + 257 per 16-bit lane (mad.lo with -1, then add.u16x2).  With stray bits 14/15 in lane 0 of
    the predictor, dd = a + pk still has the residual in its low byte, [a >= p] in bit 8, and lane 1 untouched; the
    overflow sum q + p keeps its bit 8 too."""
    def add16x2(x, y):
        return ((x + y) & 0xFFFF) | ((((x >> 16) + (y >> 16)) & 0xFFFF) << 16)
    rng = np.random.default_rng(9)
    for _ in range(20000):
        a0, a1, p0, p1, q0, q1 = (int(v) for v in rng.integers(0, 256, 6))
        stray = int(rng.integers(0, 4)) << 14
        a, p = a0 | (a1 << 16), (p0 | stray) | (p1 << 16)
        pk = add16x2((~p) & U32, 0x01010101)
        dd = (a + pk) & U32
        assert (dd & 0xFF, (dd >> 16) & 0xFF) == ((a0 - p0) & 255, (a1 - p1) & 255)
        assert ((dd >> 8) & 1, (dd >> 24) & 1) == (int(a0 >= p0), int(a1 >= p1))
        ov = ((q0 | (q1 << 16)) + p) & U32
        assert ((ov >> 8) & 1, (ov >> 24) & 1) == (int(q0 + p0 > 255), int(q1 + p1 > 255))


# ---- fp16x2 arithmetic on integer lanes (hgi_tile_swar.cuh: hfma2 / pred_pk2 / encode2) -------------------------
# A lane holding an integer n < 2048 is the fp16 number n * 2^-24; HFMA2 is modelled as an exact product and sum in
# float64 (22-bit product, < 53 bits after the add) followed by ONE rounding to fp16 (numpy: nearest even, subnormals kept).
def _h2f(bits):
    return float(np.array([bits], dtype=np.uint16).view(np.float16)[0])


def _f2h(v):
    with np.errstate(over="raise"):
        return int(np.array([v], dtype=np.float64).astype(np.float16).view(np.uint16)[0])


def hfma_lane(a, b, c):
    return _f2h(_h2f(a) * _h2f(b) + _h2f(c))


def hfma2(a, b, c):
    return hfma_lane(a & 0xFFFF, b & 0xFFFF, c & 0xFFFF) | (hfma_lane(a >> 16, b >> 16, c >> 16) << 16)


def f16_quant_constants(error):
    """quant_swar(): hK, hc1, hS, hc2 (one lane)."""
    scale = 2.0 * error + 1.0
    base = 64.0 if error == 10 else 128.0
    inv_ulp = 1024.0 / base
    return (_f2h(16777216.0 / (inv_ulp * scale)), _f2h(base + (error / scale - 0.5 + 0.5 / scale) / inv_ulp),
            _f2h(inv_ulp * scale * 2.0 ** -24), _f2h(-1024.0 * scale * 2.0 ** -24))


# H_EIGHTH .. H_257ULP belong to round 2's first predictor form (fp16_pred_pk_yb), the others to the kernel
H_EIGHTH, H_NEG_EIGHTH, H_511ULP, H_257ULP, H_255_256 = 0x3000, 0xB000, 0x01FF, 0x0101, 0x3BF8
H_QUARTER_LO, H_NEG_QUARTER_LO, H_512ULP, H_256ULP = 0x33FF, 0xB3FF, 0x0200, 0x0100


def fp16_pred_pk_yb(A, B, C, D):
    """pred_pk2<Crossed> of round 2's first fp16 form: lanes 2T + 4w + 7, times 1/8."""
    x1 = (A ^ B) & 0x00010001
    w = x1 & (C ^ D) & (A ^ C)
    yb = (2 * (A + B + C) + 2 * D + 0x00070007 + 4 * w) & U32
    assert (yb & 0xFFFF) < 2048 and (yb >> 16) < 2048          # inside the range where lane bits == value * 2^24
    rep = lambda h: h | (h << 16)
    return hfma2(yb, rep(H_EIGHTH), rep(H_511ULP)), hfma2(yb, rep(H_NEG_EIGHTH), rep(H_257ULP))


def fp16_pred_pk(A, B, C, D):
    """pred_pk2<Crossed>: (p + 512 lanes, pk lanes) from clean corner lanes: m = T + 2w, one HFMA2 by 1/4 - 2^-13."""
    va, vc = (A + B) & U32, (C + D) & U32
    w = ((A ^ C) & 0x00010001) & va & vc
    m = (va + vc + 2 * w) & U32
    assert (m & 0xFFFF) <= 1022 and (m >> 16) <= 1022
    rep = lambda h: h | (h << 16)
    return hfma2(m, rep(H_QUARTER_LO), rep(H_512ULP)), hfma2(m, rep(H_NEG_QUARTER_LO), rep(H_256ULP))


def test_fp16_constants_are_what_the_header_says():
    assert _h2f(H_EIGHTH) == 0.125 and _h2f(H_NEG_EIGHTH) == -0.125 and _h2f(H_511ULP) == 511 * 2.0 ** -24
    assert _h2f(H_257ULP) == 257 * 2.0 ** -24 and _h2f(H_255_256) == 255 / 256
    assert _h2f(H_QUARTER_LO) == 0.25 - 2.0 ** -13 and _h2f(H_NEG_QUARTER_LO) == -(0.25 - 2.0 ** -13)
    assert _h2f(H_512ULP) == 512 * 2.0 ** -24 and _h2f(H_256ULP) == 256 * 2.0 ** -24
    for n in list(range(0, 2048, 7)) + [1023, 1024, 1025, 2047]:
        assert _h2f(n) == n * 2.0 ** -24                        # subnormals and the first normal binade share the ulp


def test_fp16_divide_by_four_is_a_floor_for_every_sum():
    """RN(m * (1/4 - 2^-13) + 512) == 512 + (m + 1) // 4 and RN(256 - m * (1/4 - 2^-13)) == 256 - (m + 1) // 4 for
    every m = T + 2w the predictor can form (0..1022), and the parity term from the column sums equals the three-XOR
    form for all 16 parity patterns."""
    for m in range(0, 1023):
        assert hfma_lane(m, H_QUARTER_LO, H_512ULP) == 512 + (m + 1) // 4, m
        assert hfma_lane(m, H_NEG_QUARTER_LO, H_256ULP) == 256 - (m + 1) // 4, m
    for A, B, C, D in itertools.product((0, 1, 2, 3, 254, 255), repeat=4):
        assert (((A ^ C) & 1) & (A + B) & (C + D)) == ((A ^ B) & (C ^ D) & (A ^ C) & 1)


def fp16_pred(A, B, C, D):
    """pred2<Crossed> (decode): the same sum, RN(m * (1/4 - 2^-13)) with a zero addend -> clean lanes."""
    va, vc = (A + B) & U32, (C + D) & U32
    w = ((A ^ C) & 0x00010001) & va & vc
    rep = lambda h: h | (h << 16)
    return hfma2((va + vc + 2 * w) & U32, rep(H_QUARTER_LO), 0)


def test_fp16_decode_predictor_matches_reference():
    for m in range(0, 1023):
        assert hfma_lane(m, H_QUARTER_LO, 0) == (m + 1) // 4, m
    rng = np.random.default_rng(12)
    for v in rng.integers(0, 256, (20000, 8)):
        A, B, C, D, A2, B2, C2, D2 = (int(x) for x in v)
        args = (A | (A2 << 16), B | (B2 << 16), C | (C2 << 16), D | (D2 << 16))
        got = fp16_pred(*args)
        assert (got & 0xFFFF, got >> 16) == (ref_pred(A, B, C, D), ref_pred(A2, B2, C2, D2)) and got == swar_pred(*args)


def test_fp16_predictor_matches_reference():
    vals = [0, 1, 2, 3, 4, 5, 126, 127, 128, 129, 252, 253, 254, 255]
    for A, B, C, D in itertools.product(vals, repeat=4):
        A2, B2, C2, D2 = 255 - A, B ^ 1, (C + 77) & 255, D       # a different cell in the other lane
        r0, r1 = ref_pred(A, B, C, D), ref_pred(A2, B2, C2, D2)
        for form in (fp16_pred_pk, fp16_pred_pk_yb):
            p, pk = form(A | (A2 << 16), B | (B2 << 16), C | (C2 << 16), D | (D2 << 16))
            assert (p & 0xFFFF, p >> 16) == (r0 + 512, r1 + 512) and (pk & 0xFFFF, pk >> 16) == (256 - r0, 256 - r1)
    rng = np.random.default_rng(11)
    for v in rng.integers(0, 256, (20000, 8)):
        A, B, C, D, A2, B2, C2, D2 = (int(x) for x in v)
        p, pk = fp16_pred_pk(A | (A2 << 16), B | (B2 << 16), C | (C2 << 16), D | (D2 << 16))
        assert (p & 0xFFFF, p >> 16) == (ref_pred(A, B, C, D) + 512, ref_pred(A2, B2, C2, D2) + 512)
        assert pk == (0x03000300 - p) & U32


def test_fp16_quantizer_is_exact_for_every_residual():
    for error in (10, 20, 30):
        hK, hc1, hS, hc2 = f16_quant_constants(error)
        scale = 2 * error + 1
        for d in range(256):
            r = hfma_lane(d, hK, hc1)
            assert hfma_lane(r, hS, hc2) == ((d + error) // scale) * scale, (error, d)


def fp16_encode2(a, p, pk, error, fma_mask):
    """encode2<false, FMA_MASK>: returns (q lanes, recon lanes)."""
    hK, hc1, hS, hc2 = (h | (h << 16) for h in f16_quant_constants(error))
    dd = (a + pk) & U32
    d = dd & M16
    q = hfma2(hfma2(d, hK, hc1), hS, hc2)
    ov = (q + p) & U32
    x = (~(ov ^ dd)) & 0x01000100
    if fma_mask:                                               # 0x0100 * 255/256 == 0x00FF, exact
        m = hfma2(x, H_255_256 | (H_255_256 << 16), 0)
    else:
        m = min(x & 0xFFFF, 0xFF) | (min(x >> 16, 0xFF) << 16)
    q = (q & ~m & U32) | (dd & m)
    return q, (a + q - d) & U32


def test_fp16_encode_point_exhaustive():
    """All (a, p) pairs, every Linear level, both mask variants: symbol and reconstruction."""
    cache = {}
    for level, error in ((1, 10), (2, 20), (3, 30)):
        table, _ = oc.quant_table(oc.QUANT_LINEAR, level)
        hK, hc1, hS, hc2 = f16_quant_constants(error)
        qt = [hfma_lane(hfma_lane(d, hK, hc1), hS, hc2) for d in range(256)]     # per-lane quantizer, memoised
        for p0 in range(256):
            for a0 in range(256):
                dd = a0 + 256 - p0
                d = dd & 255
                q = qt[d]
                ov = q + p0 + 512                                # pred_pk2 hands over p + 512
                x = (~(ov ^ dd)) & 0x0100
                for m in (min(x, 0xFF), hfma_lane(x, H_255_256, 0)):
                    qq = (q & ~m) | (dd & m & 0xFFFF)
                    assert (qq, (a0 + qq - d) & 0xFFFF) == ref_encode(a0, p0, table), (level, a0, p0)
    # the two-lane form on a sample (lane independence)
    rng = np.random.default_rng(5)
    table, _ = oc.quant_table(oc.QUANT_LINEAR, 2)
    for v in rng.integers(0, 256, (3000, 4)):
        a0, a1, p0, p1 = (int(x) for x in v)
        p = p0 | (p1 << 16)
        for fm in (False, True):
            q, r = fp16_encode2(a0 | (a1 << 16), p + 0x02000200, (0x01000100 - p) & U32, 20, fm)
            assert (q & 0xFFFF, r & 0xFFFF) == ref_encode(a0, p0, table) and (q >> 16, r >> 16) == ref_encode(a1, p1, table)
