// hgi_device.cuh -- device-side primitives shared by the HGI kernels (sm_100a).
//
// Arithmetic restated from the reference (paths relative to the reference tree):
//   prediction  src/interpolator.rs:43-54 (Crossed), :19-26 (LeftTop)
//   quantizer   src/quantizator.rs:50-60 (Linear table), :27-29 (NoOp)
// Everything is u8 / small unsigned integer arithmetic; there is no floating point.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace hgi {

enum : int { kInterpCrossed = 0, kInterpLeftTop = 3 };
enum : int { kModeEncode = 0, kModeDecode = 1 };

// src/interpolator.rs:43-54.  a=(x0,y0) b=(x0,y1) c=(x1,y0) d=(x1,y1).
template <int INTERP>
__device__ __forceinline__ uint32_t predict(uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
    if (INTERP == kInterpLeftTop) return a;                 // src/interpolator.rs:26
    const uint32_t left  = (a + b + 1u) >> 1;               // :46
    const uint32_t right = (d + c + 1u) >> 1;               // :47
    const uint32_t top   = (c + a + 1u) >> 1;               // :48
    const uint32_t bot   = (d + b + 1u) >> 1;               // :49
    return (left + right + top + bot) >> 2;                 // :51 (no rounding term at HEAD)
}

// Error bound of a QuantizationLevel (src/quantizator.rs:43-48).
__host__ __device__ __forceinline__ uint32_t level_error(int quant_kind, int quant_level)
{
    return quant_kind == 0 ? 0u : 10u * (uint32_t)(quant_level & 3);
}

// table[v] of src/quantizator.rs:50-60, computed (v + e) / (2e+1) * (2e+1), truncated to u8.
__host__ __device__ __forceinline__ uint32_t quant_entry(uint32_t v, uint32_t error)
{
    const uint32_t scale = 2u * error + 1u;
    return (((v + error) / scale) * scale) & 0xFFu;
}

}  // namespace hgi
