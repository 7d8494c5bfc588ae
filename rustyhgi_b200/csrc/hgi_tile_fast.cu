// hgi_tile_fast.cu -- the fused HGI tile kernel (sm_100a), register-prefetch variant: it runs every pass of every
// plane.  The pass/tile/halo decomposition is the one tests/tile_model.py states plainly, restructured so the work per
// pixel is ~4x below a byte-wise formulation (shared device code: hgi_tile_swar.cuh):
//
//  * every level s in {2,4,8,16} of the tile lives in its own DENSE shared-memory plane P_s (lattice-s points
//    only, one byte each), so each level is "the finest level of a half-size image": even rows read
//    [R a R a ...], odd rows [a a a a ...] -- natural 16-bit-lane SWAR;
//  * a level reads its corners (and the coarser symbols) from the coarser plane P_2s / Q_2s and writes complete
//    words into P_s / Q_s, so no separate "insert" step exists;
//  * the finest level never touches shared memory for pixels: each thread loads its own 16x2-pixel units with
//    128-bit global loads at kernel start (a software prefetch that is in flight while the coarse levels run)
//    and stores finished grid / image words straight to HBM;
//  * two pixels per 32-bit register: predictor, residuals, the Linear quantizer (an exact multiply-shift, checked
//    on the host against src/quantizator.rs:50-60 for all 256 inputs) and the overflow fix-up
//    (src/encoder.rs:56-60) are all 16-bit-lane SWAR, with adds and interleaves steered to the FMA pipe because
//    the ALU pipe (LOP3/SHF/PRMT) is the kernel's limiter;
//  * the s = 2 level is owner-computed: the thread that holds a 16x4 pixel strip runs cell row ry, words 2sx and
//    2sx+1 of that level from its registers (level2_owner) and keeps P_2 / Q_2 of the strip for the finest level;
//  * the fringe (the extra cell column / row a tile recomputes instead of exchanging) is one more word column and
//    cell row of the same SWAR loop;
//  * interior tiles (tile + halo inside the plane) run a body without any in-image predicate (EDGE = false): a
//    branch in the light kernels, a launch of its own for the quantizing encode (instruction-cache footprint);
//  * the shared-memory window base is pinned in a register (opaque_smem);
//  * EXTRA instantiations also write the reconstruction plane;
//  * instantiations: ALIGNED (row pitch % 16 == 0, 16-byte bases: 128-bit accesses; the width itself may be anything
//    when the caller pads its rows) or any pitch / base alignment (32-bit accesses, funnel-shifted when rows are not
//    4-byte aligned, bytes at the ragged right edge);
//  * a D > 1 pass (levels coarser than 16) first gathers its lattice into a dense plane (hgi_decimate_kernel, coalesced)
//    and then runs this same kernel on it: the strided in-kernel gather it replaces cost 16 us per pass on a
//    16384^2 plane against 4 us for the dense tile.
//
// Reference semantics: src/encoder.rs:39-71, src/decoder.rs:18-46, src/utils.rs:11-41,
// src/interpolator.rs:15-28,41-91, src/quantizator.rs:41-74.
// Tile shape / CTA size / residency of the register-prefetch kernel.  Measured on B200 (bench.py, 4096 frames,
// ms per step, at the time of the sweep): 128x64 tiles with 128 threads (2 units per thread) at 10 CTAs/SM 14.5;
// 128x128 / 256 / 6: 15.1; 128x64 / 256 / 8: 16.0.  Small CTAs keep every barrier inside four warps.
#include <cstdlib>
#include "hgi_tile_swar.cuh"

namespace hgi {

namespace {

#ifndef HGI_FAST_MIN_BLOCKS
#define HGI_FAST_MIN_BLOCKS 10
#endif
// the headline instantiations of decode and the identity encode fit 40 registers without spilling: 12 CTAs per SM hide more of their memory
// latency (-3.5 %, A/B); the quantizing encode is 1.6 % slower that way and the EXTRA variants would spill
#ifndef HGI_FAST_MIN_BLOCKS_LIGHT
#define HGI_FAST_MIN_BLOCKS_LIGHT 12
#endif

// 16-pixel chunk I/O.  ALIGNED (w % 16 == 0, 16-byte-aligned bases): one 128-bit access, `nvalid` is 0 or 16.
// Otherwise (any width / alignment): complete chunks use 32-bit accesses -- directly when the address is
// 4-byte aligned, else five aligned loads funnel-shifted into place (`may_overread` says the 1..3 bytes after the
// chunk are still inside the plane batch) / aligned middle words plus byte head and tail for stores; ragged chunks
// at the right image edge use byte accesses.  Bytes beyond the image read as 0 and are never written.
// Zero the bytes of an aligned chunk that lie in the row padding (nvalid..15).  Deliberately not inlined, see load_chunk.
__device__ __noinline__ uint4 mask_padding(uint4 a, int nvalid)   // by value: arguments and result travel in registers
{
    const uint32_t nb = (uint32_t)min(nvalid, 16);
    a.x &= nb >= 4 ? 0xFFFFFFFFu : ((1u << (8 * nb)) - 1u);
    a.y &= nb >= 8 ? 0xFFFFFFFFu : (nb <= 4 ? 0u : ((1u << (8 * (nb - 4))) - 1u));
    a.z &= nb >= 12 ? 0xFFFFFFFFu : (nb <= 8 ? 0u : ((1u << (8 * (nb - 8))) - 1u));
    a.w &= nb >= 16 ? 0xFFFFFFFFu : (nb <= 12 ? 0u : ((1u << (8 * (nb - 12))) - 1u));
    return a;
}

// `ragged` (CTA-uniform, from the launch arguments): rows are padded and the width is not a multiple of 16, so an
// ALIGNED chunk may hold padding; with whole-chunk rows the masking code is skipped by a uniform branch.
template <bool ALIGNED>
__device__ __forceinline__ uint4 load_chunk(const uint8_t* __restrict__ ptr, int nvalid, bool may_overread, bool ragged)
{
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (nvalid <= 0) return v;
    if (ALIGNED) {
        // padded rows: the chunk is in memory as a whole, bytes beyond the image are the caller's padding -> read as 0
        uint4 a = __ldg(reinterpret_cast<const uint4*>(ptr));
        if (ragged) a = mask_padding(a, nvalid);   // a call the compiler cannot predicate: whole-chunk planes skip it with one branch
        return a;
    }
    const uint32_t sh = (uint32_t)((uintptr_t)ptr & 3u);
    if (nvalid >= 16 && (sh == 0 || may_overread)) {
        const uint32_t* q = reinterpret_cast<const uint32_t*>(ptr - sh);
        const uint32_t w0 = __ldg(q), w1 = __ldg(q + 1), w2 = __ldg(q + 2), w3 = __ldg(q + 3);
        if (sh == 0) return make_uint4(w0, w1, w2, w3);
        const uint32_t w4 = __ldg(q + 4), s8 = 8 * sh;
        return make_uint4(__funnelshift_r(w0, w1, s8), __funnelshift_r(w1, w2, s8), __funnelshift_r(w2, w3, s8),
                          __funnelshift_r(w3, w4, s8));
    }
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int i = 0; i < 16; ++i)
        if (i < nvalid) w[i >> 2] |= (uint32_t)__ldg(ptr + i) << (8 * (i & 3));
    return make_uint4(w[0], w[1], w[2], w[3]);
}

template <bool ALIGNED>
__device__ __forceinline__ void store_chunk(uint8_t* __restrict__ ptr, const uint32_t (&w)[4], int nvalid)
{
    if (nvalid <= 0) return;
    if (ALIGNED) {
        *reinterpret_cast<uint4*>(ptr) = make_uint4(w[0], w[1], w[2], w[3]);
        return;
    }
    const uint32_t sh = (uint32_t)((uintptr_t)ptr & 3u);
    if (nvalid >= 16 && sh == 0) {
        uint32_t* q = reinterpret_cast<uint32_t*>(ptr);
        q[0] = w[0]; q[1] = w[1]; q[2] = w[2]; q[3] = w[3];
    } else if (nvalid >= 16) {
        // head: 4 - sh bytes up to the next aligned address, three aligned words, tail: sh bytes
        const uint32_t hb = 4u - sh, s8 = 8 * hb;
        for (uint32_t i = 0; i < hb; ++i) ptr[i] = (uint8_t)(w[0] >> (8 * i));
        uint32_t* q = reinterpret_cast<uint32_t*>(ptr + hb);
        q[0] = __funnelshift_r(w[0], w[1], s8);
        q[1] = __funnelshift_r(w[1], w[2], s8);
        q[2] = __funnelshift_r(w[2], w[3], s8);
        for (uint32_t i = 0; i < sh; ++i) ptr[12 + hb + i] = (uint8_t)(w[3] >> (8 * (hb + i)));
    } else {
#pragma unroll
        for (int i = 0; i < 16; ++i)
            if (i < nvalid) ptr[i] = (uint8_t)(w[i >> 2] >> (8 * (i & 3)));
    }
}

// sm_100 addresses shared memory through the cluster window: every basic block that touches a __shared__ object
// rebuilds its base (S2UR SR_CgaCtaId + UMOV + ULEA, 4 % of this kernel's instructions).  Passing the 32-bit shared
// address through an empty asm makes it an ordinary value the compiler keeps in a register; the accesses still
// compile to LDS/STS because the pointer is rebuilt with the shared->generic intrinsic.
__device__ __forceinline__ FastSmem& opaque_smem(FastSmem& s)
{
    uint32_t a = (uint32_t)__cvta_generic_to_shared(&s);
    asm volatile("" : "+r"(a));
    return *reinterpret_cast<FastSmem*>(__cvta_shared_to_generic(a));
}

// EDGE = 0: the tile and its whole halo lie inside the image, so every extent is a compile-time constant
// EDGE = 2: a tile of the right tile column of a plane whose width is a multiple of the tile width, in a tile row whose
//           halo rows are inside the image: exactly TW columns (no right halo), all rows -- constants again
// EDGE = 1: anything else
// and all the in-image predicates (loads, stores, fringe cells, masks) fold away.
template <int MODE, int INTERP, bool IDENTITY, bool EXTRA, int NLEV, bool ALIGNED, int EDGE>
__device__ __forceinline__ void tile_body(const PassArgs& p, FastSmem& sm, uint32_t tx, uint32_t ty)
{
    constexpr int F = 1 << NLEV;
    const int tid = threadIdx.x;
    __builtin_assume(tid >= 0 && tid < NT);     // lets the row/column range tests of interior tiles fold
    const uint32_t img = blockIdx.z;
    const uint32_t X0 = tx * TW, Y0 = ty * TH;
    const int xin = EDGE == 1 ? (int)min((uint32_t)(TW + FMAX + 1), p.w - X0) : (EDGE == 2 ? TW : TW + FMAX + 1);   // in-image extent of tile + halo
    const int yin = EDGE == 1 ? (int)min((uint32_t)(TH + FMAX + 1), p.h - Y0) : TH + FMAX + 1;
    const bool edge = EDGE != 0;
    const size_t tile_off = ((size_t)img * p.h + Y0) * p.pitch + X0;   // CTA-uniform; the same in the source and output planes
    const size_t pitch = (size_t)p.pitch;
    const uint8_t* __restrict__ tile = p.src + tile_off;
    const bool top = (p.c_recon == nullptr);
    const bool ragged = EDGE == 1 && ALIGNED && p.vec_ok == 2u;   // padded rows whose width is not a multiple of 16
    const QuantSwar qc = {p.q_one, p.q_mul, p.q_add, p.q_shift, p.q_scale, p.q_rmask, p.q_qmul, p.q_hK, p.q_hc1, p.q_hS, p.q_hc2};   // filled by the launcher

#ifdef HGI_VAR_POISON_SMEM
    // Debug variant (tools/build_variant.sh poisonXX -DHGI_VAR_POISON_SMEM=0xXX): the planes start as a known
    // pattern instead of whatever the previous CTA left.  The kernel is allowed to COMPUTE on unstaged bytes (the
    // fringe words reach two columns / one row past anything a consumer reads) but no such byte may reach an output:
    // the parity suite must pass unchanged for every pattern -- the stand-in for `compute-sanitizer --tool
    // initcheck` on shared memory, which is closed on this pool (profiles/r02_sanitizer.md).
    for (int i = tid; i < (int)(sizeof(FastSmem) / 4); i += NT)
        reinterpret_cast<uint32_t*>(&sm)[i] = 0x01010101u * (uint32_t)(HGI_VAR_POISON_SMEM);
    __syncthreads();
#endif
    // ---- 1. global loads: this thread's NU 16x2-pixel units (kept in registers for the finest level) ----
    const int sx = tid & 7, ry = tid >> 3;          // 8 column strips x RPB thread rows, NU adjacent row pairs each
    const int nvalid = max(0, min(16, xin - 16 * sx));   // in-image bytes of this thread's chunks (0 or 16 if ALIGNED)
    // a thread's NU units are vertically adjacent row pairs (rp = NU*ry + u): the corner row between two units is
    // unpacked once and shared (A/B measured ~3 % faster than units RPB row pairs apart)
    const uint32_t toff = (uint32_t)(2 * NU * ry) * p.pitch + (uint32_t)(16 * sx);   // tile-relative, fits 32 bits (pitch < 2^26)
    uint4 ev[NU], od[NU];
#pragma unroll
    for (int u = 0; u < NU; ++u) {
        const int y = 2 * (NU * ry + u);
        // a complete chunk may be over-read by <= 3 bytes unless it ends the very last row of the batch
        const bool last0 = EDGE != 0 && (img + 1 == gridDim.z) && (Y0 + (uint32_t)y + 1 >= p.h) && (X0 + 16u * sx + 16u >= p.pitch);
        const bool last1 = EDGE != 0 && (img + 1 == gridDim.z) && (Y0 + (uint32_t)y + 2 >= p.h) && (X0 + 16u * sx + 16u >= p.pitch);
        ev[u] = load_chunk<ALIGNED>(tile + toff + (uint32_t)(2 * u) * p.pitch, y < yin ? nvalid : 0, !last0, ragged);
        od[u] = load_chunk<ALIGNED>(tile + toff + (uint32_t)(2 * u + 1) * p.pitch, y + 1 < yin ? nvalid : 0, !last1, ragged);
    }

    // L2 prefetch for a CTA that starts about one residency later (quantizing encode only, see launch_fast_n): one
    // 128-byte line per tile row.  The bounds are CTA-uniform and evaluated by the launcher, so the other kernels and
    // the edge bodies carry nothing.  (Also prefetching the halo rows TH, TH+4, TH+8, TH+16 measured no gain.)
    if (EDGE == 0 && MODE == kModeEncode && !IDENTITY && img < p.pf_zlim && ty < p.pf_ylim) {
        if (tid < TH) {
            const uint8_t* pf = p.pf_src + tile_off + (uint32_t)tid * p.pitch;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(pf));
        }
    }

    // halo chunks (right of / below the tile) feed only the coarse planes: TH/2 right-halo chunks (rows 0,2,..,TH-2;
    // column TW) + rows TH, TH+4, TH+8 (chunks 0..8).  Two ways to fetch and stage them, chosen per kernel by A/B
    // (2048 frames, same box): spread over the upper half of the CTA, one chunk per thread (decode 1.258 ms, encode
    // Medium 1.681, encode Lossless 1.274), or all on the LAST WARP, NRIGHT/32 + 1 chunks per lane, so that the other
    // warps skip the block with one uniform branch (1.266 / 1.722 / 1.242): the identity encode takes the second.
    constexpr bool HALO_WARP = (MODE == kModeEncode) && IDENTITY;
    constexpr int NRIGHT = TH / 2, NHALO = NRIGHT + 27, NRL = NRIGHT / 32;
    // -- spread form
    const int hj = tid - (NT - 64);
    int hy = 2 * hj, hc = 8;
    bool halo = false;
    uint4 hv = make_uint4(0u, 0u, 0u, 0u);
    // -- last-warp form
    const bool halo_warp = HALO_WARP && NLEV > 1 && tid >= NT - 32;
    const int hl = tid - (NT - 32);                     // lane of the halo warp
    uint4 hvr[NRL], hvb = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int k = 0; k < NRL; ++k) hvr[k] = make_uint4(0u, 0u, 0u, 0u);
    int hyb = TH, hcb = 0;
    bool has_b = false;
    if (!HALO_WARP) {
        if (hj >= NRIGHT) {
            const int r = (hj - NRIGHT) / 9;
            hc = (hj - NRIGHT) - 9 * r;
            hy = TH + 4 * r;
        }
        halo = NLEV > 1 && hj >= 0 && hj < NHALO;
        if (halo && hy < yin)
            hv = load_chunk<ALIGNED>(tile + (uint32_t)hy * p.pitch + (uint32_t)(16 * hc), min(16, xin - 16 * hc), false, ragged);
    } else if (halo_warp) {
#pragma unroll
        for (int k = 0; k < NRL; ++k) {
            const int y = 2 * (hl + 32 * k);
            if (y < yin) hvr[k] = load_chunk<ALIGNED>(tile + (uint32_t)y * p.pitch + (uint32_t)TW, min(16, xin - TW), false, ragged);
        }
        if (hl < 27) {
            const int r = (hl >= 9) + (hl >= 18);
            has_b = true;
            hcb = hl - 9 * r;
            hyb = TH + 4 * r;
            if (hyb < yin) hvb = load_chunk<ALIGNED>(tile + (uint32_t)hyb * p.pitch + (uint32_t)(16 * hcb), min(16, xin - 16 * hcb), false, ragged);
        }
    }

    // ---- 2. stage the dense coarse planes + the coarse lattice of this pass ---------------------
    constexpr bool OWN2 = F >= 4;   // the s = 2 level runs from this thread's registers (level2_owner)
#pragma unroll
    for (int u = 0; u < NU; ++u) stage_chunk<F, OWN2>(sm.P, ev[u], 2 * (NU * ry + u), sx);
    if (halo) stage_chunk<F>(sm.P, hv, hy, hc);
    if (halo_warp) {
#pragma unroll
        for (int k = 0; k < NRL; ++k) stage_chunk<F>(sm.P, hvr[k], 2 * (hl + 32 * k), 8);
        if (has_b) stage_chunk<F>(sm.P, hvb, hyb, hcb);
    }
    if (NLEV == 4 && top) {
        // top pass with step-16 seeds (src/encoder.rs:26-37 / src/decoder.rs:22-28): the seed of lattice point
        // (16*ci, 16*cj) is byte 0 of a chunk some thread already holds; only x = TW+16 and y = TH+16 need a load
        constexpr int pf = plane_pitch(16);
        uint8_t* Pf = sm.P + plane_off(16);
        uint8_t* Qf = sm.Q + plane_off(16);
#pragma unroll
        for (int u = 0; u < NU; ++u) {
            const int y = 2 * (NU * ry + u);
            if ((y & 15) == 0) {
                Pf[(y >> 4) * pf + sx] = (uint8_t)ev[u].x;
                if (MODE == kModeEncode) Qf[(y >> 4) * pf + sx] = (uint8_t)ev[u].x;
            }
        }
        if (halo && (hy & 15) == 0 && hy <= TH) {
            Pf[(hy >> 4) * pf + hc] = (uint8_t)hv.x;
            if (MODE == kModeEncode) Qf[(hy >> 4) * pf + hc] = (uint8_t)hv.x;
        }
        if (halo_warp) {   // seeds at column TW (rows that are multiples of 16) and on row TH
#pragma unroll
            for (int k = 0; k < NRL; ++k) {
                const int y = 2 * (hl + 32 * k);
                if ((y & 15) == 0) {
                    Pf[(y >> 4) * pf + 8] = (uint8_t)hvr[k].x;
                    if (MODE == kModeEncode) Qf[(y >> 4) * pf + 8] = (uint8_t)hvr[k].x;
                }
            }
            if (has_b && hyb == TH) {
                Pf[(TH >> 4) * pf + hcb] = (uint8_t)hvb.x;
                if (MODE == kModeEncode) Qf[(TH >> 4) * pf + hcb] = (uint8_t)hvb.x;
            }
        }
        constexpr int last_ci = TW / 16 + 1, last_cj = TH / 16 + 1;
        if (tid < last_ci + last_cj + 1) {
            const int ci = tid <= last_cj ? last_ci : tid - (last_cj + 1);
            const int cj = tid <= last_cj ? tid : last_cj;
            const int x = ci * 16, y = cj * 16;
            uint8_t rv = 0;
            if (x < xin && y < yin) rv = __ldg(tile + (size_t)y * pitch + (size_t)x);
            Pf[cj * pf + ci] = rv;
            if (MODE == kModeEncode) Qf[cj * pf + ci] = rv;
        }
    } else {
        constexpr int ncx = TW / F + 2, ncy = TH / F + 2;
        constexpr int pf = plane_pitch(F);
        uint8_t* Pf = sm.P + plane_off(F);
        uint8_t* Qf = sm.Q + plane_off(F);
        for (int it = tid; it < ncx * ncy; it += NT) {
            const int cj = it / ncx, ci = it - cj * ncx;
            const int x = ci * F, y = cj * F;
            uint8_t rv = 0, qv = 0;
            if (x < xin && y < yin) {
                if (top) {   // src/encoder.rs:26-37 / src/decoder.rs:22-28: the seed is the source byte
                    rv = __ldg(tile + (size_t)y * pitch + (size_t)x);
                    qv = rv;
                } else {
                    const size_t co = ((size_t)img * p.ch + ((Y0 + y) >> NLEV)) * p.cpitch + ((X0 + x) >> NLEV);
                    rv = __ldg(p.c_recon + co);
                    if (MODE == kModeEncode) qv = __ldg(p.c_q + co);
                }
            }
            Pf[cj * pf + ci] = rv;
            if (MODE == kModeEncode) Qf[cj * pf + ci] = qv;
        }
    }
    __syncthreads();

    // ---- 3. coarse levels of the pass, s = F/2 .. 2 ---------------------------------------------
    if (F >= 16) coarse_level<MODE, INTERP, IDENTITY, 8>(sm, tid, qc, edge, xin, yin);
    if (F >= 8) coarse_level<MODE, INTERP, IDENTITY, 4>(sm, tid, qc, edge, xin, yin);
    uint32_t p2e[2] = {0u, 0u}, p2o[2] = {0u, 0u}, q2e[2] = {0u, 0u}, q2o[2] = {0u, 0u};
    if (OWN2) {
        level2_owner<MODE, INTERP, IDENTITY>(sm, ev[0], ev[1], sx, ry, qc, edge, xin, yin, p2e, p2o, q2e, q2o);
        coarse_level<MODE, INTERP, IDENTITY, 2, false>(sm, tid, qc, edge, xin, yin);   // fringe cells + barrier
    }

    // ---- 4. finest level: registers + P_2 / Q_2 -> HBM -------------------------------------------
    uint8_t* __restrict__ out = (MODE == kModeEncode ? p.grid_out : p.recon_out) + tile_off;
    uint32_t A[4], B[4], C[4], D[4];
    {
        const uint8_t* P2r = sm.P + plane_off(2) + (NU * ry) * plane_pitch(2) + 8 * sx;
        const uint2 ctw = OWN2 ? make_uint2(p2e[0], p2e[1]) : *reinterpret_cast<const uint2*>(P2r);
        const uint32_t cte = P2r[8];
        A[0] = lanes01(ctw.x); A[1] = lanes23(ctw.x); A[2] = lanes01(ctw.y); A[3] = lanes23(ctw.y);
        C[0] = lanes12(ctw.x); C[1] = __funnelshift_r(A[1], A[2], 16); C[2] = lanes12(ctw.y); C[3] = __funnelshift_r(A[3], cte, 16);
    }
#pragma unroll
    for (int u = 0; u < NU; ++u) {
        const int rp = NU * ry + u;
        const bool row0_ok = 2 * rp < yin, row1_ok = 2 * rp + 1 < yin;
        const uint32_t uoff = toff + (uint32_t)(2 * u) * p.pitch;
        if (u > 0) {
#pragma unroll
            for (int k = 0; k < 4; ++k) { A[k] = B[k]; C[k] = D[k]; }
        }
        {
            const uint8_t* P2r = sm.P + plane_off(2) + (rp + 1) * plane_pitch(2) + 8 * sx;
            const uint2 cbw = (OWN2 && u == 0) ? make_uint2(p2o[0], p2o[1]) : *reinterpret_cast<const uint2*>(P2r);
            const uint32_t cbe = P2r[8];
            B[0] = lanes01(cbw.x); B[1] = lanes23(cbw.x); B[2] = lanes01(cbw.y); B[3] = lanes23(cbw.y);
            D[0] = lanes12(cbw.x); D[1] = __funnelshift_r(B[1], B[2], 16); D[2] = lanes12(cbw.y); D[3] = __funnelshift_r(B[3], cbe, 16);
        }
        const uint32_t evw[4] = {ev[u].x, ev[u].y, ev[u].z, ev[u].w};
        const uint32_t odw[4] = {od[u].x, od[u].y, od[u].z, od[u].w};
        uint32_t out_ev[4], out_od[4], rec_ev[4], rec_od[4];
        uint2 qcw = make_uint2(0u, 0u);
        if (MODE == kModeEncode)
            qcw = OWN2 ? (u == 0 ? make_uint2(q2e[0], q2e[1]) : make_uint2(q2o[0], q2o[1]))
                       : *reinterpret_cast<const uint2*>(sm.Q + plane_off(2) + rp * plane_pitch(2) + 8 * sx);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t a1 = lanes_odd(evw[k]), a2 = lanes_even(odw[k]), a3 = lanes_odd(odw[k]);
            if (MODE == kModeEncode) {
                uint32_t q[3], r[3];
                encode_cells<INTERP, IDENTITY>(A[k], B[k], C[k], D[k], a1, a2, a3, qc, q, r);
                const uint32_t qw = (k < 2) ? qcw.x : qcw.y;
                out_ev[k] = pack_even_row(qw, q[0], (k & 1) != 0);
                out_od[k] = pack_sym<IDENTITY>(q[1], q[2]);
                if (EXTRA) {
                    rec_ev[k] = interleave(A[k], r[0]);
                    rec_od[k] = interleave(r[1], r[2]);
                }
            } else {
                const uint32_t pr = pred2<INTERP>(A[k], B[k], C[k], D[k], qc.one);
                out_ev[k] = pack_lo(A[k], decode2(a1, pr, qc.one));
                out_od[k] = pack_lo(decode2(a2, pr, qc.one), decode2(a3, pr, qc.one));
            }
        }
        store_chunk<ALIGNED>(out + uoff, out_ev, row0_ok ? nvalid : 0);
        store_chunk<ALIGNED>(out + uoff + p.pitch, out_od, row1_ok ? nvalid : 0);
        if (MODE == kModeEncode && EXTRA) {
            if (p.recon_out != nullptr) {
                uint8_t* __restrict__ rout = p.recon_out + tile_off;
                store_chunk<ALIGNED>(rout + uoff, rec_ev, row0_ok ? nvalid : 0);
                store_chunk<ALIGNED>(rout + uoff + p.pitch, rec_od, row1_ok ? nvalid : 0);
            }
        }
    }
}

template <int MODE, int INTERP, bool IDENTITY, bool EXTRA, int NLEV, bool ALIGNED>
__global__ void __launch_bounds__(NT, (IDENTITY && !EXTRA && ALIGNED && NLEV == 4) ? HGI_FAST_MIN_BLOCKS_LIGHT : HGI_FAST_MIN_BLOCKS)
hgi_tile_fast_kernel(const PassArgs p)
{
    __shared__ FastSmem sm_static;
    FastSmem& sm = opaque_smem(sm_static);
    // interior tiles (88 % of a 1080p plane) take the predicate-free body; only the headline instantiations of the
    // light kernels are split this way -- the quantizing encode is split at launch level instead (below): with both
    // bodies in one kernel its code is 43 KB and it runs 12 % slower, an instruction-cache effect
    constexpr bool kSplit = ((MODE == kModeDecode) || IDENTITY) && ALIGNED && NLEV == 4;
    if (kSplit) {
        const bool interior = blockIdx.x < p.fast_itx && blockIdx.y < p.fast_ity;   // the launcher's counts of interior tile columns / rows
        if (interior) {
            tile_body<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 0>(p, sm, blockIdx.x, blockIdx.y);
            return;
        }
        // the right tile column of a plane whose width is a multiple of the tile width: constant extents again (EDGE = 2;
        // 6 % of the tiles of a 1080p frame at the interior body's ~400 instructions per warp instead of the general
        // edge body's ~810: -0.7 % per light kernel in power-capped runs, nothing at full clock where they are DRAM-bound)
        if (p.fast_rcol != 0u && blockIdx.x == p.fast_itx && blockIdx.y < p.fast_ity) {
            tile_body<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 2>(p, sm, blockIdx.x, blockIdx.y);
            return;
        }
    }
    tile_body<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 1>(p, sm, blockIdx.x, blockIdx.y);
}

// The same pass as three launches with two-dimensional tile grids (no index arithmetic in the kernel):
// PART 1 = the interior tiles [0, fast_itx) x [0, fast_ity) with the predicate-free body;
// PART 2 = the right tile columns [fast_itx, tiles_x) of the interior tile rows, general edge body;
// PART 4 = the same when there is ONE right column and it is exactly TW wide (width % TW == 0): constants again;
// PART 3 = the bottom tile rows [fast_ity, tiles_y), all columns, general edge body.
template <int MODE, int INTERP, bool IDENTITY, bool EXTRA, int NLEV, bool ALIGNED, int PART>
__global__ void __launch_bounds__(NT, (IDENTITY && !EXTRA && ALIGNED && NLEV == 4) ? HGI_FAST_MIN_BLOCKS_LIGHT : HGI_FAST_MIN_BLOCKS)
hgi_tile_fast_part_kernel(const PassArgs p)
{
    __shared__ FastSmem sm_static;
    FastSmem& sm = opaque_smem(sm_static);
    if (PART == 1) tile_body<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 0>(p, sm, blockIdx.x, blockIdx.y);
    else if (PART == 2) tile_body<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 1>(p, sm, p.fast_itx + blockIdx.x, blockIdx.y);
    else if (PART == 4) tile_body<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 2>(p, sm, p.fast_itx + blockIdx.x, blockIdx.y);
    else tile_body<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 1>(p, sm, blockIdx.x, p.fast_ity + blockIdx.y);
}

// below this many tiles (about four waves of 10 CTAs on 148 SMs) the second launch costs more than the edge predicates
// (HGI_B200_SPLIT_MIN=<tiles> overrides, a tuning hook)
inline uint64_t split_min_tiles()
{
    static const uint64_t v = [] { const char* e = getenv("HGI_B200_SPLIT_MIN"); return e ? (uint64_t)atoll(e) : (uint64_t)(4 * 1480); }();
    return v;
}

// One counted launch (hgi_ctx_kernel_launches) of a fast tile kernel.
inline void launch_one(void (*kernel)(PassArgs), dim3 nb, cudaStream_t stream, const PassArgs& a)
{
    kernel<<<nb, NT, 0, stream>>>(a);
    ++launch_count();
}

template <int MODE, int INTERP, bool IDENTITY, bool EXTRA, int NLEV, bool ALIGNED>
cudaError_t launch_fast_split(PassArgs& a, uint32_t tiles_x, uint32_t tiles_y, cudaStream_t stream)
{
    if (a.fast_itx == 0 || a.fast_ity == 0) a.fast_itx = a.fast_ity = 0;
    // the edge launches depend on nothing the interior launch writes: fork them onto the side stream when there is one
    const bool fork = a.fast_itx && a.side_stream && a.ev_fork && a.ev_join;
    cudaStream_t es = fork ? a.side_stream : stream;
    if (fork) {
        cudaError_t e = cudaEventRecord(a.ev_fork, stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(a.side_stream, a.ev_fork, 0);
        if (e != cudaSuccess) return e;
    }
    if (a.fast_itx)
        launch_one(hgi_tile_fast_part_kernel<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 1>, dim3(a.fast_itx, a.fast_ity, a.n_images),
                   stream, a);
    const uint32_t ncr = tiles_x - a.fast_itx, nbr = tiles_y - a.fast_ity;
    if (ncr && a.fast_ity)     // right tile columns of the interior tile rows
        launch_one(ncr == 1 && a.w == tiles_x * (uint32_t)TW ? hgi_tile_fast_part_kernel<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 4>
                                                            : hgi_tile_fast_part_kernel<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 2>,
                   dim3(ncr, a.fast_ity, a.n_images), es, a);
    if (nbr)                   // bottom tile rows
        launch_one(hgi_tile_fast_part_kernel<MODE, INTERP, IDENTITY, EXTRA, NLEV, ALIGNED, 3>, dim3(tiles_x, nbr, a.n_images), es, a);
    if (fork) {
        cudaError_t e = cudaEventRecord(a.ev_join, a.side_stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, a.ev_join, 0);
        if (e != cudaSuccess) return e;
    }
    return cudaGetLastError();
}

// One grid of a pass: `a` holds the slice's planes -- its images, or one image from the slice's first tile row down, so
// that a.h still covers the halo rows below the slice -- and `rows` the slice's tile rows (gridDim.y).
template <int MODE, int INTERP, int NLEV, bool ALIGNED>
cudaError_t launch_fast_slice(PassArgs a, uint32_t tiles_x, uint32_t rows, cudaStream_t stream)
{
    // interior tile columns / rows (tile + halo inside the plane), for the bodies without in-image predicates
    const uint32_t itx = a.w >= (uint32_t)(FMAX + 1) ? min(tiles_x, (a.w - (FMAX + 1)) / TW) : 0u;
    const uint32_t ity = a.h >= (uint32_t)(FMAX + 1) ? min(rows, (a.h - (FMAX + 1)) / TH) : 0u;
    // L2 prefetch distance of the interior tiles of the quantizing encode, in residencies (148 SMs x 10 CTAs): that
    // kernel is bound by its instruction stream, so the DRAM latency of a tile's first loads is the one stall it cannot
    // cover with other work; fetching the tile into L2 about one residency earlier takes it away (-2..3 %, A/B sweep:
    // k = 0.5..2 alike, beyond k = 2.5 the lines are evicted before use and the kernel loses 8 %).  The DRAM-bound light
    // kernels lose with any distance (+20 % at k = 2) and do not carry the code.  HGI_B200_PREFETCH=<k> overrides, 0 = off.
    static const double pf_k = [] { const char* e = getenv("HGI_B200_PREFETCH"); return e ? atof(e) : 1.0; }();
    const double pf_tiles = pf_k * 1480.0;
    const uint64_t tiles_img = (uint64_t)tiles_x * rows;
    uint32_t pf_images = 0, pf_rows = 0;
    if (pf_tiles > 0.0) {
        if ((double)tiles_img <= pf_tiles) pf_images = (uint32_t)((pf_tiles + (double)tiles_img - 1.0) / (double)tiles_img);
        else pf_rows = (uint32_t)((pf_tiles + (double)tiles_x - 1.0) / (double)tiles_x);
    }
    a.fast_itx = itx;
    a.fast_ity = ity;
    a.fast_rcol = (itx + 1 == tiles_x && a.w == tiles_x * (uint32_t)TW) ? 1u : 0u;   // ONE right column, exactly TW wide
    const bool extra = (a.recon_out != nullptr);
    // a large slice of the quantizing encode runs as split launches (interior / edges); only their interior-only
    // CTAs prefetch.  Small slices: one launch, less latency
    const bool split = MODE == kModeEncode && a.quant_error != 0 && ALIGNED && NLEV == 4 &&
                       tiles_img * a.n_images >= split_min_tiles();
    // prefetch bounds against this slice's grid: planes [0, n - pf_images) / interior tile rows [0, ity - pf_rows)
    const uint32_t zi = split ? pf_images : 0u, zr = split ? pf_rows : 0u;
    a.pf_zlim = zi ? (a.n_images > zi ? a.n_images - zi : 0u) : (zr ? a.n_images : 0u);
    a.pf_ylim = zr ? (ity > zr ? ity - zr : 0u) : 0xFFFFFFFFu;
    a.pf_src = a.src + ((uint64_t)zi * a.h + (uint64_t)zr * TH) * a.pitch;
    const dim3 nb(tiles_x, rows, a.n_images);
    if (MODE == kModeDecode) {
        launch_one(hgi_tile_fast_kernel<kModeDecode, INTERP, true, false, NLEV, ALIGNED>, nb, stream, a);
    } else if (a.quant_error == 0) {
        launch_one(!extra ? hgi_tile_fast_kernel<kModeEncode, INTERP, true, false, NLEV, ALIGNED>
                          : hgi_tile_fast_kernel<kModeEncode, INTERP, true, true, NLEV, ALIGNED>, nb, stream, a);
    } else if (split) {
        if constexpr (MODE == kModeEncode && ALIGNED && NLEV == 4) {
            const cudaError_t es = extra ? launch_fast_split<kModeEncode, INTERP, false, true, NLEV, ALIGNED>(a, tiles_x, rows, stream)
                                         : launch_fast_split<kModeEncode, INTERP, false, false, NLEV, ALIGNED>(a, tiles_x, rows, stream);
            if (es != cudaSuccess) return es;
        }
    } else {
        launch_one(!extra ? hgi_tile_fast_kernel<kModeEncode, INTERP, false, false, NLEV, ALIGNED>
                          : hgi_tile_fast_kernel<kModeEncode, INTERP, false, true, NLEV, ALIGNED>, nb, stream, a);
    }
    return cudaGetLastError();
}

// gridDim.y and gridDim.z hold at most 65535 tile rows and images: a pass runs in slices of up to 65535 whole images or,
// for a plane of more than 65535 tile rows, one image at a time in bands of up to 65535 tile rows (the kernel steps
// from image to image by h * pitch, so a band must be the only image of its grid).
template <int MODE, int INTERP, int NLEV, bool ALIGNED>
cudaError_t launch_fast_n(const PassArgs& args, cudaStream_t stream)
{
    const uint32_t tiles_x = (args.w + TW - 1) / TW, tiles_y = (args.h + TH - 1) / TH;
    if (tiles_x == 0 || tiles_y == 0 || args.n_images == 0) return cudaSuccess;
    const size_t plane = (size_t)args.pitch * args.h, cplane = (size_t)args.cpitch * args.ch;
    const uint32_t per = tiles_y <= 65535u ? 65535u : 1u;
    for (uint32_t first = 0; first < args.n_images; first += per) {
        for (uint32_t ty0 = 0; ty0 < tiles_y; ty0 += 65535u) {
            const size_t y0 = (size_t)ty0 * TH, off = (size_t)first * plane + y0 * args.pitch;
            const size_t coff = (size_t)first * cplane + (y0 >> NLEV) * args.cpitch;   // y0 is a multiple of 2^NLEV
            PassArgs a = args;
            a.n_images = args.n_images - first < per ? args.n_images - first : per;
            a.h = args.h - (uint32_t)y0;
            a.src = args.src + off;
            if (args.grid_out) a.grid_out = args.grid_out + off;
            if (args.recon_out) a.recon_out = args.recon_out + off;
            if (args.c_recon) {
                a.c_recon = args.c_recon + coff;
                a.ch = args.ch - (uint32_t)(y0 >> NLEV);
            }
            if (args.c_q) a.c_q = args.c_q + coff;
            const cudaError_t e = launch_fast_slice<MODE, INTERP, NLEV, ALIGNED>(a, tiles_x, min(65535u, tiles_y - ty0), stream);
            if (e != cudaSuccess) return e;
        }
    }
    return cudaSuccess;
}

template <int MODE, int INTERP>
cudaError_t launch_fast_t(const PassArgs& args_in, cudaStream_t stream)
{
    PassArgs a = args_in;
    fill_quant_args(a);
    if (a.d_log2 > 0) {   // coarse pass: gather the lattice into a dense plane, then an ordinary pass on it -> compact outputs
        const cudaError_t e = launch_decimate(a.src, a.pitch, a.h, a.d_log2, a.wD, a.hD, a.dpitch, a.n_images, a.dec_in, stream);
        if (e != cudaSuccess) return e;
        PassArgs v = a;
        v.src = a.dec_in;
        v.w = a.wD;
        v.h = a.hD;
        v.pitch = a.dpitch;
        v.grid_out = a.s_q;
        v.recon_out = a.s_recon;
        v.d_log2 = 0;
        v.vec_ok = (a.wD & 15u) ? 2u : 1u;   // dpitch is a 16-byte multiple and the scratch planes are cudaMalloc'ed
        a = v;
    }
    if (a.vec_ok) {
        switch (a.nlev) {
            case 1: return launch_fast_n<MODE, INTERP, 1, true>(a, stream);
            case 2: return launch_fast_n<MODE, INTERP, 2, true>(a, stream);
            case 3: return launch_fast_n<MODE, INTERP, 3, true>(a, stream);
            case 4: return launch_fast_n<MODE, INTERP, 4, true>(a, stream);
            default: return cudaErrorInvalidValue;
        }
    }
    switch (a.nlev) {   // any pitch / alignment
        case 1: return launch_fast_n<MODE, INTERP, 1, false>(a, stream);
        case 2: return launch_fast_n<MODE, INTERP, 2, false>(a, stream);
        case 3: return launch_fast_n<MODE, INTERP, 3, false>(a, stream);
        case 4: return launch_fast_n<MODE, INTERP, 4, false>(a, stream);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace

// Host-side proof obligation for the SWAR quantizer: it must equal the reference table for all
// 256 residuals at every QuantizationLevel (src/quantizator.rs:50-60).
bool quant_swar_self_check()
{
    for (uint32_t e = 10; e <= 30; e += 10) {
        const QuantSwar q = quant_swar(e);
        for (uint32_t d0 = 0; d0 < 256; ++d0) {
            const uint32_t d1 = 255u - d0;
            const uint32_t d = d0 | (d1 << 16);
            const uint32_t t = d * q.mul + q.add;
            const uint32_t v = (uint32_t)(((unsigned long long)(t & q.rmask) * q.qmul) >> 32);
            if ((v & 0xFFFFu) != quant_entry(d0, e) || (v >> 16) != quant_entry(d1, e)) return false;
        }
    }
    return true;
}

namespace {
// dst[img][y][x] = src[img][y << d][x << d] for the lattice of a D = 2^d pass; one 32-bit word (four lattice points)
// per thread, rows padded with zeros up to dpitch.  A warp reads 128 points 2^d bytes apart: at d = 4 that is every
// sector of a 2 KB run, i.e. the DRAM traffic is the image rows the lattice lives on (1/16 of the plane), coalesced.
__global__ void __launch_bounds__(256)
hgi_decimate_kernel(const uint8_t* __restrict__ src, uint32_t pitch, uint32_t h, uint32_t d, uint32_t wD, uint32_t hD,
                    uint32_t dpitch, uint8_t* __restrict__ dst)
{
    const uint32_t wx = blockIdx.x * blockDim.x + threadIdx.x;      // word index in the row
    const uint32_t y = blockIdx.y, img = blockIdx.z;
    if (wx * 4u >= dpitch) return;
    const uint8_t* row = src + ((size_t)img * h + ((size_t)y << d)) * pitch;
    uint32_t v = 0u;
#pragma unroll
    for (uint32_t i = 0; i < 4; ++i) {
        const uint32_t x = wx * 4u + i;
        if (x < wD) v |= (uint32_t)__ldg(row + ((size_t)x << d)) << (8 * i);
    }
    *reinterpret_cast<uint32_t*>(dst + ((size_t)img * hD + y) * dpitch + 4u * wx) = v;
}
}  // namespace

cudaError_t launch_decimate(const uint8_t* src, uint32_t pitch, uint32_t h, uint32_t d_log2, uint32_t wD, uint32_t hD,
                            uint32_t dpitch, uint32_t n_images, uint8_t* dst, cudaStream_t stream)
{
    if (wD == 0 || hD == 0 || n_images == 0) return cudaSuccess;
    const uint32_t words = dpitch / 4, bx = words < 256u ? ((words + 31u) / 32u) * 32u : 256u;
    // slices of up to 65535 images x 65535 rows (gridDim.z / gridDim.y); the kernel uses h and hD as plane strides only
    for (uint32_t first = 0; first < n_images; first += 65535u) {
        const uint32_t cnt = n_images - first < 65535u ? n_images - first : 65535u;
        for (uint32_t y0 = 0; y0 < hD; y0 += 65535u) {
            const dim3 nb((words + bx - 1) / bx, min(65535u, hD - y0), cnt);
            hgi_decimate_kernel<<<nb, bx, 0, stream>>>(src + ((size_t)first * h + ((size_t)y0 << d_log2)) * pitch, pitch, h,
                                                       d_log2, wD, hD, dpitch, dst + ((size_t)first * hD + y0) * dpitch);
            ++launch_count();
        }
    }
    return cudaGetLastError();
}

uint64_t& launch_count()
{
    static thread_local uint64_t n = 0;
    return n;
}

cudaError_t launch_tile_pass(int mode, int interp, const PassArgs& a, cudaStream_t stream)
{
    if (mode == kModeEncode)
        return interp == kInterpLeftTop ? launch_fast_t<kModeEncode, kInterpLeftTop>(a, stream)
                                        : launch_fast_t<kModeEncode, kInterpCrossed>(a, stream);
    return interp == kInterpLeftTop ? launch_fast_t<kModeDecode, kInterpLeftTop>(a, stream)
                                    : launch_fast_t<kModeDecode, kInterpCrossed>(a, stream);
}

}  // namespace hgi
