// hgi_tile_swar.cuh -- shared device code of the fast HGI tile kernels (sm_100a): dense per-level plane
// geometry, 16-bit-lane SWAR arithmetic (predictor, quantizer, fix-up), plane staging and the coarse-level
// routines of hgi_tile_fast.cu (register-prefetch kernel, 128x64 tiles, 128 threads).
//
// Reference semantics: src/encoder.rs:39-71, src/decoder.rs:18-46, src/utils.rs:11-41,
// src/interpolator.rs:15-28,41-91, src/quantizator.rs:41-74.
#pragma once
#include "hgi_device.cuh"
#include "hgi_kernels.h"

namespace hgi {
namespace {

constexpr int TW = 128;                  // tile width  (lattice points)
constexpr int TH = 64;                   // tile height
constexpr int NT = 128;                  // threads per CTA
constexpr int NU = TH * 4 / NT;          // 16x2-pixel units per thread in the finest level
constexpr int RPB = NT / 8;              // row pairs covered by one unit block (8 column strips x RPB row pairs)
constexpr int NWARPS = NT / 32;
constexpr int FMAX = 1 << kMaxPassLevels;
constexpr uint32_t M16 = 0x00FF00FFu;

static_assert(TW == 128 && NU == 2 && NU * NT == TH * 4, "thread mapping assumes 128x64 tiles, two units per thread");

// Dense level planes.  P_s holds lattice-s points of the tile + halo: columns 0..TW/s+1,
// rows 0..TH/s+1 (the last ones are only partially needed, see fringe_cell).
__host__ __device__ constexpr int plane_pitch(int s) { return s == 2 ? 96 : (s == 4 ? 48 : (s == 8 ? 32 : 16)); }
__host__ __device__ constexpr int plane_rows(int s) { return TH / s + 2; }
__host__ __device__ constexpr int plane_bytes(int s) { return plane_rows(s) * plane_pitch(s); }
__host__ __device__ constexpr int plane_off(int s)
{
    return s == 2 ? 0 : (s == 4 ? plane_bytes(2) : (s == 8 ? plane_bytes(2) + plane_bytes(4)
                                                               : plane_bytes(2) + plane_bytes(4) + plane_bytes(8)));
}
constexpr int PLANE_BYTES = plane_bytes(2) + plane_bytes(4) + plane_bytes(8) + plane_bytes(16);  // 4544

// Highest tile-relative coordinate at which a new point of sub-step s is still needed (see DESIGN.md 4.1):
// TW-1, TW, TW+s for s = 1, 2, >= 4.  Used as compile-time constants in fringe_cell().

// ---- 16-bit-lane SWAR primitives (two pixels per register) -----------------------------------
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) { return __byte_perm(a, b, sel); }
// bytes (i, i+1) of w -> lanes
__device__ __forceinline__ uint32_t lanes01(uint32_t w) { return prmt(w, 0u, 0x4140u); }
__device__ __forceinline__ uint32_t lanes12(uint32_t w) { return prmt(w, 0u, 0x4241u); }
__device__ __forceinline__ uint32_t lanes23(uint32_t w) { return prmt(w, 0u, 0x4342u); }
// bytes (0,2) / (1,3) of w -> lanes
__device__ __forceinline__ uint32_t lanes_even(uint32_t w) { return w & M16; }
__device__ __forceinline__ uint32_t lanes_odd(uint32_t w) { return prmt(w, 0u, 0x4341u); }
// lanes (lo0, lo1), (hi0, hi1) -> bytes lo0 hi0 lo1 hi1
__device__ __forceinline__ uint32_t interleave(uint32_t even_lanes, uint32_t odd_lanes)
{
    // odd * 256 + even as ONE multiply-add: it issues on the FMA pipe, the ALU pipe is the kernel's bottleneck
    uint32_t r;
    asm("mad.lo.u32 %0, %1, 256, %2;" : "=r"(r) : "r"(odd_lanes), "r"(even_lanes));
    return r;
}
// Low bytes of the lanes, interleaved: bytes even.l0 odd.l0 even.l1 odd.l1.  Unlike interleave() the inputs may
// carry junk above bit 7 of each lane (9-bit sums), so the "& 0x00FF00FF" of a wrapping add costs nothing.
__device__ __forceinline__ uint32_t pack_lo(uint32_t even_lanes, uint32_t odd_lanes)
{
    return prmt(even_lanes, odd_lanes, 0x6240u);
}
// symbols of encode2<IDENTITY>: dirty lanes when IDENTITY (-> pack_lo), clean otherwise (-> interleave on the FMA pipe)
template <bool IDENTITY>
__device__ __forceinline__ uint32_t pack_sym(uint32_t even_lanes, uint32_t odd_lanes)
{
    return IDENTITY ? pack_lo(even_lanes, odd_lanes) : interleave(even_lanes, odd_lanes);
}
// Symbols of an even row: bytes [c0, q0, c1, q1] where c0/c1 are two consecutive bytes of the coarser level's symbol
// word `qw` (bytes 0,1 or, if `hi`, bytes 2,3) and q0/q1 the low bytes of the lanes of `odd_lanes` -- one PRMT instead
// of unpacking the coarser symbols into lanes and interleaving.
__device__ __forceinline__ uint32_t pack_even_row(uint32_t qw, uint32_t odd_lanes, bool hi)
{
    return prmt(qw, odd_lanes, hi ? 0x6342u : 0x6140u);
}
// a + b issued as a multiply-add (x * 1 + y): same result, but on the FMA pipe instead of the saturated ALU pipe
// `one` is a register that holds 1 but is opaque to ptxas (it comes from the kernel arguments); with a literal 1
// ptxas folds the multiply-add back into IADD3 on the ALU pipe.
__device__ __forceinline__ uint32_t fadd(uint32_t a, uint32_t b, uint32_t one)
{
    uint32_t r;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(one), "r"(b));
    return r;
}
// ---- fp16x2 arithmetic on integer lanes ------------------------------------------------------------------------
// A 16-bit lane that holds an integer n < 2048 is, read as an fp16 bit pattern, the number n * 2^-24 (subnormals and
// the first normal binade share the ulp 2^-24; sm_100 does not flush them).  HFMA2 therefore does exact integer
// arithmetic on both lanes of a register with ONE rounding to the nearest integer at the end -- which turns a
// "multiply, add, shift" (three instructions, the shift on the saturated ALU pipe) into one instruction on the FMA
// pipe, and yields clean lanes (no bits shifted across the lane boundary).  tools/ubench_pipes.cu measures the
// pipes (HFMA2 / IMAD: FMA pipe, 0.5 per clock; LOP3 / PRMT / SHF / VIMNMX / HSET2: ALU pipe, 0.5 per clock; IMAD.HI
// 0.25 per clock) and checks the exactness on the device; tests/test_swar_model.py models it on the CPU.
__device__ __forceinline__ uint32_t hfma2(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}
__device__ __forceinline__ uint32_t hmul2(uint32_t a, uint32_t b)
{
    uint32_t r;
    asm("mul.rn.f16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    return r;
}
constexpr uint32_t kH_255_256 = 0x3BF83BF8u;      // 255/256: 0x0100 -> 0x00FF per lane

// Crossed predictor for the quantizing encode: returns pk = 256 - pred per lane and, if WANT_P, p = pred + 512 (the
// only consumer is bit 8 of q + p; the bias keeps the lane away from -0 when pred == 0); both clean.
// pred = (T + 1 + 2w) >> 2 (see pred2 below) = floor((m + 1) / 4) with m = T + 2w <= 1022 (w = 1 needs mixed
// parities, i.e. T <= 1018).  One HFMA2 divides and floors: with b = 1/4 - 2^-13 (fp16 0x33FF) the exact product is
// m/4 - m/8192 = k + {-1/4, 0, 1/4, 1/2} - eps for m = 4k + {-1, 0, 1, 2}, 0 <= eps < 1/8 (eps > 0 whenever m > 0), so it
// lies strictly inside (k - 3/8, k + 1/2): round-to-nearest gives k and never sees a tie.  pred + 512 = RN(m b + 512),
// 256 - pred = RN(256 - m b).  The parity term needs only two LOP3: the parities of A^B and C^D are those of the
// column sums A + B and C + D, which the sum needs anyway: w = ((A ^ C) & 1) & (A + B) & (C + D).
// (Round 2, first form: lanes 2T + 4w + 7 times 1/8 -- one multiply-add, one constant move and one LOP3 more.)
constexpr uint32_t kH_quarter_lo = 0x33FF33FFu;   // 1/4 - 2^-13
constexpr uint32_t kH_neg_quarter_lo = 0xB3FFB3FFu;
constexpr uint32_t kH_512ulp = 0x02000200u;
constexpr uint32_t kH_256ulp = 0x01000100u;
template <int INTERP, bool WANT_P>
__device__ __forceinline__ uint32_t pred_pk2(uint32_t A, uint32_t B, uint32_t C, uint32_t D, uint32_t one, uint32_t& p)
{
    if (INTERP == kInterpLeftTop) {                                            // src/interpolator.rs:26
        p = A;
        uint32_t pk;
        asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(pk) : "r"(A), "r"(0u - one), "r"(0x01000100u));
        return pk;
    }
    const uint32_t va = fadd(A, B, one), vc = fadd(C, D, one);                 // column sums, lanes <= 510
    const uint32_t w = ((A ^ C) & 0x00010001u) & va & vc;                      // two LOP3
    uint32_t m = fadd(va, vc, one);                                            // T
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(m) : "r"(w), "r"(one + one), "r"(m));   // T + 2w <= 1022
    if (WANT_P) p = hfma2(m, kH_quarter_lo, kH_512ulp);
    return hfma2(m, kH_neg_quarter_lo, kH_256ulp);
}

// src/interpolator.rs:43-54 per lane.  With avg(x,y) = (x+y+1)>>1 = (x + y + ((x^y)&1)) / 2, the sum of the
// four edge averages is T + E/2, T = A+B+C+D, where E counts the edges of the cycle A-B-D-C-A whose
// endpoints differ in parity (0, 2 or 4).  Working through floor((T + E/2)/4) by the parity of T gives
//     pred = (((T + 1) >> 1) + w) >> 1,    w = (A^B) & (C^D) & (A^C) & 1
// (E/2 only matters when it makes T+E/2 cross a multiple of 4: T odd -> the +1; T = 2 mod 4 with all
// three parity tests true -> the w).  Checked against the four-average form in tests/test_swar_model.py.
// pred == (T + 1 + 2w) >> 2, computed with the division of pred_pk2: RN(m (1/4 - 2^-13)) with m = T + 2w.  Clean
// lanes; 2 ALU-pipe and 5 FMA-pipe operations per register (two cells) instead of 16 for the four averages.
template <int INTERP>
__device__ __forceinline__ uint32_t pred2(uint32_t A, uint32_t B, uint32_t C, uint32_t D, uint32_t one)
{
    if (INTERP == kInterpLeftTop) return A;                                    // src/interpolator.rs:26
    const uint32_t va = fadd(A, B, one), vc = fadd(C, D, one);
    const uint32_t w = ((A ^ C) & 0x00010001u) & va & vc;
    uint32_t m = fadd(va, vc, one);
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(m) : "r"(w), "r"(one + one), "r"(m));
    return hfma2(m, kH_quarter_lo, 0u);
}

// Linear quantizer as an exact per-lane multiply-shift: ((d + e) / scale) * scale for d in 0..255.
struct QuantSwar {
    uint32_t one;           // the constant 1, opaque to the compiler (see fadd)
    uint32_t mul, add, shift, scale;
    uint32_t rmask, qmul;   // q = umulhi(t & rmask, qmul): rmask = 0xF << shift per lane, qmul = scale << (32 - shift)
    // fp16x2 form (both lanes): r = d * hK + hc1 = base + floor((d + e) / scale) * ulp(base), q = r * hS + hc2
    uint32_t hK, hc1, hS, hc2;
};
// double -> fp16 bits, round to nearest even, subnormals included (host side; |v| < 65520)
__host__ inline uint32_t f16_bits(double v)
{
    const uint32_t sign = v < 0 ? 0x8000u : 0u;
    const double a = v < 0 ? -v : v;
    if (a == 0) return sign;
    int e;
    (void)frexp(a, &e);                       // a = f * 2^e, f in [0.5, 1)
    int E = e - 1;                            // a = 1.m * 2^E
    if (E < -14) {                            // subnormal: multiples of 2^-24
        const uint32_t m = (uint32_t)nearbyint(ldexp(a, 24));
        return sign | m;                      // m == 1024 is the smallest normal, same encoding
    }
    uint32_t m = (uint32_t)nearbyint(ldexp(a, 10 - E));   // in [1024, 2048]
    if (m == 2048u) { m = 1024u; ++E; }
    return sign | ((uint32_t)(E + 15) << 10) | (m - 1024u);
}
__host__ inline double f16_value(uint32_t b)
{
    const int e = (b >> 10) & 31, m = b & 1023;
    const double x = e ? ldexp(1.0 + m / 1024.0, e - 15) : ldexp(m / 1024.0, -14);
    return (b & 0x8000u) ? -x : x;
}
__host__ __device__ inline QuantSwar quant_swar(uint32_t error)   // the fp16 constants are filled on the host only
{
    // (k, c, n) with ((x*k + c) >> n) == x / (2e+1) for all x in [e, 255+e] and x*k + c < 2^16
    uint32_t k = 0, c = 0, n = 0;
    if (error == 10) { k = 195; c = 195; n = 12; }
    else if (error == 20) { k = 25; c = 0; n = 10; }
    else if (error == 30) { k = 67; c = 67; n = 12; }
    QuantSwar q;
    q.one = 1;
    q.mul = k;
    q.add = (error * k + c) * 0x00010001u;
    q.shift = n;
    q.scale = 2 * error + 1;
    q.rmask = (0xFu << n) * 0x00010001u;
    q.qmul = n ? (q.scale << (32 - n)) : 0u;
    q.hK = q.hc1 = q.hS = q.hc2 = 0u;
#ifndef __CUDA_ARCH__
    if (error) {
        // r = base + floor((d + e) / scale) / inv_ulp with base = 128 (ulp 1/8); e = 10 needs base = 64 (ulp 1/16)
        // because 2^24 / (8 * 21) is not a finite fp16.  The offset 0.5 / scale centres the quotient between two
        // multiples of 1 / scale, so the rounding of r never sees a tie: RN == floor.
        const double scale = 2.0 * error + 1.0, base = error == 10 ? 64.0 : 128.0, inv_ulp = 1024.0 / base;
        q.hK = f16_bits(16777216.0 / (inv_ulp * scale)) * 0x00010001u;
        q.hc1 = f16_bits(base + (error / scale - 0.5 + 0.5 / scale) / inv_ulp) * 0x00010001u;
        q.hS = f16_bits(ldexp(inv_ulp * scale, -24)) * 0x00010001u;
        q.hc2 = f16_bits(-ldexp(1024.0 * scale, -24)) * 0x00010001u;
    }
#endif
    return q;
}

// the launchers evaluate the constants on the host, once per launch
__host__ inline void fill_quant_args(PassArgs& a)
{
    const QuantSwar q = quant_swar(a.quant_error);
    a.q_one = q.one; a.q_mul = q.mul; a.q_add = q.add; a.q_shift = q.shift; a.q_scale = q.scale; a.q_rmask = q.rmask; a.q_qmul = q.qmul;
    a.q_hK = q.hK; a.q_hc1 = q.hc1; a.q_hS = q.hS; a.q_hc2 = q.hc2;
}

// src/encoder.rs:52-64 for two pixels.  Returns the symbols; `recon` = what the decoder rebuilds.
// p, pk = 256 - p: clean lanes (pred_pk2).  Quantizer (src/quantizator.rs:50-60) on the FMA pipe: two HFMA2, see
// QuantSwar; the lanes of q come out as plain integers.
// FMA_MASK: the fix-up mask is built on the FMA pipe (HMUL2) instead of the ALU pipe (VIMNMX).
template <bool IDENTITY, bool FMA_MASK>
__device__ __forceinline__ uint32_t encode2(uint32_t a, uint32_t p, uint32_t pk, const QuantSwar& qc, uint32_t& recon)
{
    const uint32_t dd = fadd(a, pk, qc.one);          // per lane a + 256 - p: low byte = the residual, bit 8 = [a >= p]
    if (IDENTITY) {
        recon = a;                                    // p + (a - p) == a
        return dd;                                    // low byte of each lane = the symbol; packed with pack_lo()
    }
    const uint32_t d = dd & M16;                      // :53 wrapping_sub
    const uint32_t r = hfma2(d, qc.hK, qc.hc1);       // base + floor((d + e) / scale) * ulp
    uint32_t q = hfma2(r, qc.hS, qc.hc2);             // :54 table[d]
    const uint32_t ov = fadd(q, p, qc.one);           // bit 8 = overflow (p may carry the bias 512)  (:56)
    // overflow_is_expected = [a < p] = !bit8(dd)  =>  mismatch iff bit8(ov) == bit8(dd)       (:57-58)
    const uint32_t x = ~(ov ^ dd) & 0x01000100u;
    uint32_t m;                                       // 0x00FF in every mismatching lane
    if (FMA_MASK) m = hmul2(x, kH_255_256);           // 256 ulp * 255/256, exact
    else asm("min.u16x2 %0, %1, %2;" : "=r"(m) : "r"(x), "r"(0x00FF00FFu));
    q = (q & ~m) | (dd & m);                          // :59 (m only covers the low byte of a lane, so dd's flag bit drops out: one LOP3)
    // :63 (p + q) mod 256.  p + d == a (mod 256) and, once the fix-up has run, a + (q - d) stays inside 0..255
    // (that is exactly what the overflow test guards), so the lanes need neither a borrow nor a mask.
    recon = a + q - d;
    return q;
}
// the three new points of a cell pair (a1: even row, a2 / a3: odd row)
template <int INTERP, bool IDENTITY>
__device__ __forceinline__ void encode_cells(uint32_t A, uint32_t B, uint32_t C, uint32_t D, uint32_t a1, uint32_t a2, uint32_t a3,
                                             const QuantSwar& qc, uint32_t (&q)[3], uint32_t (&r)[3])
{
    uint32_t p = 0u;
    const uint32_t pk = pred_pk2<INTERP, !IDENTITY>(A, B, C, D, qc.one, p);
    // two of the three fix-up masks on the FMA pipe balance it best against the ALU pipe (profiles/r02_fast_tile_kernel.md)
    q[0] = encode2<IDENTITY, true>(a1, p, pk, qc, r[0]);
    q[1] = encode2<IDENTITY, true>(a2, p, pk, qc, r[1]);
    q[2] = encode2<IDENTITY, false>(a3, p, pk, qc, r[2]);
}

// src/decoder.rs:39 for two pixels; the low byte of each lane is the pixel (pack with pack_lo())
__device__ __forceinline__ uint32_t decode2(uint32_t g, uint32_t p, uint32_t one) { return fadd(p, g, one); }

__device__ __forceinline__ uint32_t valid_mask(int col0, int row, int xin_s, int yin_s)
{
    const int n = xin_s - col0;
    if (row >= yin_s || n <= 0) return 0u;
    return n >= 4 ? 0xFFFFFFFFu : ((1u << (8 * n)) - 1u);
}

struct FastSmem {
    alignas(16) uint8_t P[PLANE_BYTES];   // encode: pixels -> reconstruction; decode: residuals -> pixels
    alignas(16) uint8_t Q[PLANE_BYTES];   // encode: residual symbols
};

// Stage one 16-byte chunk (columns 16c..16c+15 of tile row y, y even) into the dense planes of the
// levels that are computed in this pass (s < F).  c == 8 is the right-halo chunk (x = TW..TW+15).
// SKIP2: the chunk's owner runs the s = 2 level from its registers (level2_owner), so P_2 needs no staging.
template <int F, bool SKIP2 = false>
__device__ __forceinline__ void stage_chunk(uint8_t* P, const uint4 v, int y, int c)
{
    if (F > 2 && !SKIP2 && y <= TH) {
        uint8_t* row = P + plane_off(2) + (y >> 1) * plane_pitch(2);
        if (c < 8)
            *reinterpret_cast<uint2*>(row + 8 * c) = make_uint2(prmt(v.x, v.y, 0x6420u), prmt(v.z, v.w, 0x6420u));
        else
            row[64] = (uint8_t)v.x;
    }
    if (F > 4 && (y & 3) == 0 && y <= TH + 4) {
        uint8_t* row = P + plane_off(4) + (y >> 2) * plane_pitch(4);
        if (c < 8)
            *reinterpret_cast<uint32_t*>(row + 4 * c) = prmt(prmt(v.x, v.y, 0x0040u), prmt(v.z, v.w, 0x0040u), 0x5410u);
        else
            *reinterpret_cast<uint16_t*>(row + 32) = (uint16_t)prmt(v.x, v.y, 0x0040u);
    }
    if (F > 8 && (y & 7) == 0 && y <= TH + 8) {
        uint8_t* row = P + plane_off(8) + (y >> 3) * plane_pitch(8);
        *reinterpret_cast<uint16_t*>(row + 2 * c) = (uint16_t)prmt(v.x, v.z, 0x0040u);
    }
}

// One word (two cells, four plane columns) of a coarse level s >= 2, SWAR.
template <int MODE, int INTERP, bool IDENTITY, int S>
__device__ __forceinline__ void level_word(FastSmem& sm, int g, int cy, const QuantSwar& qc, bool edge,
                                           int xin_s, int yin_s)
{
    constexpr int ps = plane_pitch(S), pc = plane_pitch(2 * S);
    uint8_t* Ps = sm.P + plane_off(S);
    const uint8_t* Pc = sm.P + plane_off(2 * S);
    const uint8_t* ct = Pc + cy * pc + 2 * g;
    // three corner bytes per row as a 16-bit and an 8-bit load (zero-extended): their zero bytes serve as the lane
    // padding, so the two registers need not be merged first
    const uint32_t tlo = *reinterpret_cast<const uint16_t*>(ct), thi = ct[2];
    const uint32_t blo = *reinterpret_cast<const uint16_t*>(ct + pc), bhi = ct[pc + 2];
    const uint32_t A = prmt(tlo, thi, 0x3120u), C = prmt(tlo, thi, 0x3421u), B = prmt(blo, bhi, 0x3120u), D = prmt(blo, bhi, 0x3421u);
    uint32_t* pev = reinterpret_cast<uint32_t*>(Ps + (2 * cy) * ps + 4 * g);
    uint32_t* pod = reinterpret_cast<uint32_t*>(Ps + (2 * cy + 1) * ps + 4 * g);
    const uint32_t ev = *pev, od = *pod;
    const uint32_t a1 = lanes_odd(ev), a2 = lanes_even(od), a3 = lanes_odd(od);   // clean lanes: the sums must stay < 2^16
    uint32_t r[3];
    if (MODE == kModeEncode) {
        uint32_t q[3];
        encode_cells<INTERP, IDENTITY>(A, B, C, D, a1, a2, a3, qc, q, r);
        uint8_t* Qs = sm.Q + plane_off(S);
        const uint8_t* Qc = sm.Q + plane_off(2 * S);
        const uint32_t qcw = (uint32_t)*reinterpret_cast<const uint16_t*>(Qc + cy * pc + 2 * g);
        *reinterpret_cast<uint32_t*>(Qs + (2 * cy) * ps + 4 * g) = pack_even_row(qcw, q[0], false);
        *reinterpret_cast<uint32_t*>(Qs + (2 * cy + 1) * ps + 4 * g) = pack_sym<IDENTITY>(q[1], q[2]);
    } else {
        const uint32_t p = pred2<INTERP>(A, B, C, D, qc.one);
        r[0] = decode2(a1, p, qc.one);
        r[1] = decode2(a2, p, qc.one);
        r[2] = decode2(a3, p, qc.one);
    }
    uint32_t wev, wod;
    if (MODE == kModeDecode) { wev = pack_lo(A, r[0]); wod = pack_lo(r[1], r[2]); }   // r = p + g with carry bits
    else { wev = interleave(A, r[0]); wod = interleave(r[1], r[2]); }               // encode: recon lanes are clean
    if (edge) {   // out-of-image reconstruction must read as 0 (src/interpolator.rs:75-82)
        wev &= valid_mask(4 * g, 2 * cy, xin_s, yin_s);
        wod &= valid_mask(4 * g, 2 * cy + 1, xin_s, yin_s);
    }
    *pev = wev;
    *pod = wod;
}

// The s = 2 level of one thread's own strip, from registers: the thread that holds image rows 4*ry .. 4*ry+3,
// columns 16*sx .. 16*sx+15 (r0 = row 4*ry, r1 = row 4*ry+2) owns cell row ry, words 2*sx and 2*sx+1 of the s = 2
// plane.  Same arithmetic as level_word<.., 2>, but the pixels never visit shared memory, the two words share their
// corner loads, and the results stay in registers for the finest level (p2e/p2o = P_2 rows 2*ry, 2*ry+1;
// q2e/q2o = the symbols of those rows, encode only); only the reconstruction is stored, for the neighbours.
template <int MODE, int INTERP, bool IDENTITY>
__device__ __forceinline__ void level2_owner(FastSmem& sm, const uint4& r0, const uint4& r1, int sx, int ry,
                                             const QuantSwar& qc, bool edge, int xin, int yin,
                                             uint32_t (&p2e)[2], uint32_t (&p2o)[2], uint32_t (&q2e)[2], uint32_t (&q2o)[2])
{
    constexpr int ps = plane_pitch(2), pc = plane_pitch(4);
    const int xin_s = (int)(((uint32_t)xin + 1) / 2u), yin_s = (int)(((uint32_t)yin + 1) / 2u);
    const uint8_t* ct = sm.P + plane_off(4) + ry * pc + 4 * sx;
    const uint32_t ctw = *reinterpret_cast<const uint32_t*>(ct), cte = ct[4];
    const uint32_t cbw = *reinterpret_cast<const uint32_t*>(ct + pc), cbe = ct[pc + 4];
    uint32_t qcw = 0u;
    if (MODE == kModeEncode) qcw = *reinterpret_cast<const uint32_t*>(sm.Q + plane_off(4) + ry * pc + 4 * sx);
    const uint32_t evw[2] = {prmt(r0.x, r0.y, 0x6420u), prmt(r0.z, r0.w, 0x6420u)};   // lattice-2 points of row 4*ry
    const uint32_t odw[2] = {prmt(r1.x, r1.y, 0x6420u), prmt(r1.z, r1.w, 0x6420u)};   // ... of row 4*ry+2
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const uint32_t A = k ? lanes23(ctw) : lanes01(ctw), C = k ? prmt(ctw, cte, 0x5453u) : lanes12(ctw);
        const uint32_t B = k ? lanes23(cbw) : lanes01(cbw), D = k ? prmt(cbw, cbe, 0x5453u) : lanes12(cbw);
        const uint32_t a1 = lanes_odd(evw[k]), a2 = lanes_even(odw[k]), a3 = lanes_odd(odw[k]);
        uint32_t r[3];
        if (MODE == kModeEncode) {
            uint32_t q[3];
            encode_cells<INTERP, IDENTITY>(A, B, C, D, a1, a2, a3, qc, q, r);
            q2e[k] = pack_even_row(qcw, q[0], k != 0);
            q2o[k] = pack_sym<IDENTITY>(q[1], q[2]);
        } else {
            const uint32_t p = pred2<INTERP>(A, B, C, D, qc.one);
            r[0] = decode2(a1, p, qc.one);
            r[1] = decode2(a2, p, qc.one);
            r[2] = decode2(a3, p, qc.one);
        }
        uint32_t wev, wod;
        if (MODE == kModeDecode) { wev = pack_lo(A, r[0]); wod = pack_lo(r[1], r[2]); }
        else { wev = interleave(A, r[0]); wod = interleave(r[1], r[2]); }
        if (edge) {   // out-of-image reconstruction must read as 0 (src/interpolator.rs:75-82)
            wev &= valid_mask(8 * sx + 4 * k, 2 * ry, xin_s, yin_s);
            wod &= valid_mask(8 * sx + 4 * k, 2 * ry + 1, xin_s, yin_s);
        }
        p2e[k] = wev;
        p2o[k] = wod;
    }
    uint8_t* row = sm.P + plane_off(2) + (2 * ry) * ps + 8 * sx;
    *reinterpret_cast<uint2*>(row) = make_uint2(p2e[0], p2e[1]);
    *reinterpret_cast<uint2*>(row + ps) = make_uint2(p2o[0], p2o[1]);
}

// One fringe word of the s = 2 level, reduced to the ONE point per cell the finest level reads (see fringe_cell): the
// words of the fringe row (it < wpr: cell row TH/4) need their (x0+1, y0) points -- plane row TH/2, all of which the
// last row of finest cells reads as its lower corners -- and the words of the fringe column (cell column TW/4) the
// (x0, y0+1) point of their first cell -- plane column TW/2, the right corners of the last finest cell column.  One
// code path for both (the 32 words share a warp): the point pair comes from the even-row word (bytes 1, 3) or from the
// odd-row word (bytes 0, 2) by address and PRMT selector, one encode2 / decode2 instead of three, no symbols (the
// symbols of fringe points are never output).  The even-row word is rebuilt as [A r A r]; in a column word the r
// bytes land on plane columns TW/2 + 1, + 3 and the odd-row word carries r in its lanes (byte 0 = the point, bytes
// 1..3 = lane padding / the second cell): nobody reads those.
template <int MODE, int INTERP, bool IDENTITY>
__device__ __forceinline__ void fringe2_word(FastSmem& sm, int it, const QuantSwar& qc, bool edge, int xin_s, int yin_s)
{
    constexpr int ps = plane_pitch(2), pc = plane_pitch(4), wpr = TW / 8, ncy = TH / 4;
    const bool is_row = it < wpr;
    const int g = is_row ? it : wpr, cy = is_row ? ncy : it - wpr;
    const uint8_t* ct = sm.P + plane_off(4) + cy * pc + 2 * g;
    // three corner bytes per row as a 16-bit and an 8-bit load (zero-extended): their zero bytes serve as the lane
    // padding, so the two registers need not be merged first
    const uint32_t tlo = *reinterpret_cast<const uint16_t*>(ct), thi = ct[2];
    const uint32_t blo = *reinterpret_cast<const uint16_t*>(ct + pc), bhi = ct[pc + 2];
    const uint32_t A = prmt(tlo, thi, 0x3120u), C = prmt(tlo, thi, 0x3421u), B = prmt(blo, bhi, 0x3120u), D = prmt(blo, bhi, 0x3421u);
    uint8_t* ev = sm.P + plane_off(2) + (2 * cy) * ps + 4 * g;
    const uint32_t w = *reinterpret_cast<const uint32_t*>(is_row ? ev : ev + ps);
    const uint32_t a = prmt(w, 0u, is_row ? 0x4341u : 0x4240u);
    uint32_t r, wev;
    if (MODE == kModeEncode) {
        uint32_t p = 0u;
        const uint32_t pk = pred_pk2<INTERP, !IDENTITY>(A, B, C, D, qc.one, p);
        (void)encode2<IDENTITY, false>(a, p, pk, qc, r);
        wev = interleave(A, r);
    } else {
        r = decode2(a, pred2<INTERP>(A, B, C, D, qc.one), qc.one);
        wev = pack_lo(A, r);
    }
    if (edge) {   // out-of-image reconstruction must read as 0 (src/interpolator.rs:75-82)
        wev &= valid_mask(4 * g, 2 * cy, xin_s, yin_s);
        r &= valid_mask(4 * g, 2 * cy + 1, xin_s, yin_s);
    }
    *reinterpret_cast<uint32_t*>(ev) = wev;
    if (!is_row) *reinterpret_cast<uint32_t*>(ev + ps) = r;
}

// One fringe cell (extra cell column / row right of and below the tile) of a coarse level, scalar.
template <int MODE, int INTERP, bool IDENTITY, int S>
__device__ __forceinline__ void fringe_cell(FastSmem& sm, int cx, int cy, const QuantSwar& qc, int xin_s, int yin_s)
{
    constexpr int ps = plane_pitch(S), pc = plane_pitch(2 * S);
    constexpr int xlim = (S == 2 ? TW : TW + S) / S, ylim = (S == 2 ? TH : TH + S) / S;   // need_limit / S
    uint8_t* Ps = sm.P + plane_off(S);
    const uint8_t* Pc = sm.P + plane_off(2 * S);
    const uint32_t A = Pc[cy * pc + cx], C = Pc[cy * pc + cx + 1];
    const uint32_t B = Pc[(cy + 1) * pc + cx], D = Pc[(cy + 1) * pc + cx + 1];
    const uint32_t pred = predict<INTERP>(A, B, C, D);
    const int x0 = 2 * cx, y0 = 2 * cy;
    Ps[y0 * ps + x0] = (uint8_t)A;   // the coarser lattice point itself (already 0 when out of image)
    const int px[3] = {x0 + 1, x0, x0 + 1};
    const int py[3] = {y0, y0 + 1, y0 + 1};
    // At S == 2 the finest level only reads column TW/2 and row TH/2 of this plane: a cell of the fringe column
    // contributes its (x0, y0+1) point, a cell of the fringe row its (x0+1, y0) point, nothing else.
    constexpr bool ONE = (S == 2);
    constexpr int NPT = ONE ? 1 : 3;
    const int k2 = (x0 == xlim) ? 1 : 0;
#pragma unroll
    for (int kk = 0; kk < NPT; ++kk) {
        const int x = ONE ? x0 + 1 - k2 : px[kk], y = ONE ? y0 + k2 : py[kk];
        if (x > xlim || y > ylim || x >= xin_s || y >= yin_s) continue;
        uint8_t* r = &Ps[y * ps + x];
        if (MODE == kModeEncode) {
            const uint32_t a = *r;
            const uint32_t diff = (a - pred) & 0xFFu;
            uint32_t q = diff;
            if (!IDENTITY) {
                q = (((diff * qc.mul + (qc.add & 0xFFFFu)) >> qc.shift) & 0xFu) * qc.scale;
                if (((pred + q) > 255u) != ((pred + diff) > 255u)) q = diff;
            }
            *r = (uint8_t)((pred + q) & 0xFFu);       // symbols of fringe points are never output
        } else {
            *r = (uint8_t)((pred + *r) & 0xFFu);
        }
    }
}

// One coarse level (sub-step S >= 2) of the tile: SWAR words over the tile's own cells on the low
// threads, the fringe cells (cell column TW/(2S), cell row TH/(2S)) on the high threads; ends with a CTA barrier.
// The fringe (cell column TW/(2S) and cell row TH/(2S), needed by the finer levels of this tile) is computed as
// ordinary SWAR words: word column `wpr` and cell row `ncy` extend the loop.  Their second cell / odd row reaches
// two plane columns (one plane row) further than any consumer reads -- inside the plane pitch, computed from stale
// bytes, never used.
// WORDS = false: only the fringe words (the caller has run the tile's own cells itself, see level2_owner).
template <int MODE, int INTERP, bool IDENTITY, int S, bool WORDS = true>
__device__ __forceinline__ void coarse_level(FastSmem& sm, int tid, const QuantSwar& qc, bool edge, int xin, int yin)
{
    constexpr int wpr = TW / (4 * S);               // SWAR words per cell row (2 cells each)
    constexpr int ncy = TH / (2 * S), ncx = TW / (2 * S);
    const int xin_s = (int)(((uint32_t)xin + S - 1) / (uint32_t)S), yin_s = (int)(((uint32_t)yin + S - 1) / (uint32_t)S);
    // the identity encode's s = 2 fringe stays scalar: one point per cell without a quantizer is ~35 instructions on
    // two warps, cheaper for that latency-bound kernel than 32 full words on one warp (A/B)
    constexpr bool kScalarFringe = !WORDS && IDENTITY && MODE == kModeEncode;
    if (kScalarFringe) {
        constexpr int nfr = (ncy + 1) + ncx;
        for (int it = NT - 1 - tid; it < nfr; it += NT) {
            const int cx = it <= ncy ? ncx : it - (ncy + 1);
            const int cy = it <= ncy ? it : ncy;
            if (2 * cx < xin_s && 2 * cy < yin_s)
                fringe_cell<MODE, INTERP, IDENTITY, S>(sm, cx, cy, qc, xin_s, yin_s);
            else
                (sm.P + plane_off(S))[(2 * cy) * plane_pitch(S) + 2 * cx] = 0;
        }
    } else if (WORDS) {
        constexpr int wx = wpr + 1, nwords = wx * (ncy + 1);
        for (int it = tid; it < nwords; it += NT) {
            const int cy = (int)((uint32_t)it / (uint32_t)wx);
            level_word<MODE, INTERP, IDENTITY, S>(sm, it - cy * wx, cy, qc, edge, xin_s, yin_s);
        }
    } else {
        // wpr words of the fringe row (cy = ncy), then ncy words of the fringe column (g = wpr), on the highest threads
        // (32 words = one warp at S = 2); of the corner cell only the lattice point itself is read by anyone: a copy of
        // the coarser plane's byte (0 when out of the image)
        constexpr int nfw = wpr + ncy;
        for (int it = NT - 1 - tid; it < nfw; it += NT) {
            if (S == 2) fringe2_word<MODE, INTERP, IDENTITY>(sm, it, qc, edge, xin_s, yin_s);
            else level_word<MODE, INTERP, IDENTITY, S>(sm, it < wpr ? it : wpr, it < wpr ? ncy : it - wpr, qc, edge, xin_s, yin_s);
        }
        if (tid == NT - 1)
            (sm.P + plane_off(S))[(2 * ncy) * plane_pitch(S) + 4 * wpr] = (sm.P + plane_off(2 * S))[ncy * plane_pitch(2 * S) + 2 * wpr];
    }
    __syncthreads();
}

}  // namespace
}  // namespace hgi
