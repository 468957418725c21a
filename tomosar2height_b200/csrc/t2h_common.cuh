// Shared device helpers for the sm_100a hot-path kernels (see include/t2h.h for the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>
#include "t2h.h"

#define T2H_CHECK_LAUNCH()                                   \
  do {                                                       \
    cudaError_t e_ = cudaPeekAtLastError();                  \
    if (e_ != cudaSuccess) { (void)cudaGetLastError(); return T2H_ERR_CUDA; } \
  } while (0)

namespace t2h {

constexpr int kWarp = 32;
constexpr int kSMs = 148;  // B200

// ---- Morton (Z-order) codes for 16-bit cell coordinates; x occupies the even bits ----------
__host__ __device__ __forceinline__ uint32_t part1by1(uint32_t v) {
  v &= 0x0000ffffu;
  v = (v | (v << 8)) & 0x00ff00ffu;
  v = (v | (v << 4)) & 0x0f0f0f0fu;
  v = (v | (v << 2)) & 0x33333333u;
  v = (v | (v << 1)) & 0x55555555u;
  return v;
}
__host__ __device__ __forceinline__ uint32_t compact1by1(uint32_t v) {
  v &= 0x55555555u;
  v = (v | (v >> 1)) & 0x33333333u;
  v = (v | (v >> 2)) & 0x0f0f0f0fu;
  v = (v | (v >> 4)) & 0x00ff00ffu;
  v = (v | (v >> 8)) & 0x0000ffffu;
  return v;
}
__host__ __device__ __forceinline__ uint32_t cell_code(uint32_t ix, uint32_t iy, int reso, int morton) {
  return morton ? (part1by1(ix) | (part1by1(iy) << 1)) : (ix + (uint32_t)reso * iy);
}
__host__ __device__ __forceinline__ void cell_decode(uint32_t code, int reso, int morton, int& ix, int& iy) {
  if (morton) { ix = (int)compact1by1(code); iy = (int)compact1by1(code >> 1); }
  else        { ix = (int)(code % (uint32_t)reso); iy = (int)(code / (uint32_t)reso); }
}

// A feature row of C floats is covered by LPR lanes x CH float4 chunks per lane; a warp
// therefore processes RPI = 32 / LPR rows per iteration.  C = 4 * LPR * CH.
template <int LPR_, int CH_>
struct RowShape {
  static constexpr int LPR = LPR_;
  static constexpr int CH = CH_;
  static constexpr int RPI = kWarp / LPR_;
  static constexpr int C = 4 * LPR_ * CH_;
};

// order-preserving map double -> unsigned 64: a < b as doubles <=> encode_f64(a) < encode_f64(b) as integers (-0.0
// sorts just below +0.0).  Integer atomicMin / atomicMax on the codes are deterministic; radix digits of the codes
// select order statistics.
__device__ __forceinline__ unsigned long long encode_f64(double v) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double decode_f64(unsigned long long e) {
  const unsigned long long b = (e & 0x8000000000000000ull) ? (e & 0x7fffffffffffffffull) : ~e;
  return __longlong_as_double((long long)b);
}

__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, const float4& v) { *reinterpret_cast<float4*>(p) = v; }
// streaming variants: data touched once (do not keep it in L1)
__device__ __forceinline__ float4 ld4_stream(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void st4_stream(float* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ float4 shfl_xor4(const float4& v, int off) {
  float4 r;
  r.x = __shfl_xor_sync(0xffffffffu, v.x, off);
  r.y = __shfl_xor_sync(0xffffffffu, v.y, off);
  r.z = __shfl_xor_sync(0xffffffffu, v.z, off);
  r.w = __shfl_xor_sync(0xffffffffu, v.w, off);
  return r;
}

// ATen GridSampler semantics for align_corners=True, padding_mode='border':
//   g = 2p - 1 ; i = ((g + 1) / 2) * (size - 1) ; clip to [0, size-1]     (alto.py:94-95)
// every step individually rounded (no FMA contraction) so the coordinate is bit-identical to ATen's.
__device__ __forceinline__ float unnormalize_border(float p, int size) {
  float g = __fsub_rn(__fmul_rn(2.0f, p), 1.0f);
  float i = __fmul_rn(__fmul_rn(__fadd_rn(g, 1.0f), 0.5f), (float)(size - 1));
  return fminf(fmaxf(i, 0.0f), (float)(size - 1));
}

// Dispatch a kernel functor over the supported channel counts (C = 4*LPR*CH).
#define T2H_DISPATCH_ROWSHAPE(C_, ...)                                              \
  switch (C_) {                                                                     \
    case 4:    { using RS = t2h::RowShape<1, 1>;  __VA_ARGS__; } break;             \
    case 8:    { using RS = t2h::RowShape<2, 1>;  __VA_ARGS__; } break;             \
    case 16:   { using RS = t2h::RowShape<4, 1>;  __VA_ARGS__; } break;             \
    case 32:   { using RS = t2h::RowShape<8, 1>;  __VA_ARGS__; } break;             \
    case 64:   { using RS = t2h::RowShape<16, 1>; __VA_ARGS__; } break;             \
    case 128:  { using RS = t2h::RowShape<32, 1>; __VA_ARGS__; } break;             \
    case 256:  { using RS = t2h::RowShape<32, 2>; __VA_ARGS__; } break;             \
    case 384:  { using RS = t2h::RowShape<32, 3>; __VA_ARGS__; } break;             \
    case 512:  { using RS = t2h::RowShape<32, 4>; __VA_ARGS__; } break;             \
    case 640:  { using RS = t2h::RowShape<32, 5>; __VA_ARGS__; } break;             \
    case 768:  { using RS = t2h::RowShape<32, 6>; __VA_ARGS__; } break;             \
    case 896:  { using RS = t2h::RowShape<32, 7>; __VA_ARGS__; } break;             \
    case 1024: { using RS = t2h::RowShape<32, 8>; __VA_ARGS__; } break;             \
    default: return T2H_ERR_UNSUPPORTED_SHAPE;                                      \
  }

}  // namespace t2h
