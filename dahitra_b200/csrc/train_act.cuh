// dahitra_b200 — storage of the per-pixel activations that cross the boundary of the training kernels (train_decoder.cu,
// train_tokens.cu): fp32, fp16 or bf16 (DH_ACT_* of include/dahitra_b200.h; fp16 / bf16 are what autocast hands over).
// Only the storage changes: values become fp32 on load, every kernel keeps its fp32 arithmetic, and 16-bit stores round to
// nearest even.  One pixel's 32 channels live in a [B][32][N] (planar, PM = false: one element per channel row, coalesced
// across the pixel threads) or [B][N][32] (pixel-major = channels_last, PM = true: 128 bytes of fp32 as eight 16-byte vectors,
// 64 bytes of fp16 / bf16 as four) tensor.
#pragma once
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <string.h>
#include <type_traits>

__device__ __forceinline__ float dh_act_f32(float v) { return v; }
__device__ __forceinline__ float dh_act_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float dh_act_f32(__nv_bfloat16 v) { return __bfloat162float(v); }

template <typename T> __device__ __forceinline__ T dh_act_from(float v);
template <> __device__ __forceinline__ float dh_act_from<float>(float v) { return v; }
template <> __device__ __forceinline__ __half dh_act_from<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 dh_act_from<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// two 16-bit values packed in one 32-bit word (lower address = .x)
template <typename T>
__device__ __forceinline__ float2 dh_act_unpack2(unsigned u) {
  if constexpr (std::is_same<T, __half>::value) {
    __half2 h; memcpy(&h, &u, 4); return __half22float2(h);
  } else {
    __nv_bfloat162 h; memcpy(&h, &u, 4); return __bfloat1622float2(h);
  }
}
template <typename T>
__device__ __forceinline__ unsigned dh_act_pack2(float a, float b) {
  unsigned u;
  if constexpr (std::is_same<T, __half>::value) {
    const __half2 h = __floats2half2_rn(a, b); memcpy(&u, &h, 4);
  } else {
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b); memcpy(&u, &h, 4);
  }
  return u;
}

template <bool PM, typename T>
__device__ __forceinline__ void dh_load_pixel(const T* __restrict__ t, int b, int n, int N, bool live, float (&v)[32]) {
  if constexpr (PM && sizeof(T) == 4) {
    const float4* p = reinterpret_cast<const float4*>(t + ((size_t)b * N + n) * 32);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const float4 w = live ? __ldg(p + q) : make_float4(0.f, 0.f, 0.f, 0.f);
      v[4 * q] = w.x; v[4 * q + 1] = w.y; v[4 * q + 2] = w.z; v[4 * q + 3] = w.w;
    }
  } else if constexpr (PM) {
    const uint4* p = reinterpret_cast<const uint4*>(t + ((size_t)b * N + n) * 32);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint4 w = live ? __ldg(p + q) : make_uint4(0u, 0u, 0u, 0u);
      const unsigned u[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = dh_act_unpack2<T>(u[i]);
        v[8 * q + 2 * i] = f.x; v[8 * q + 2 * i + 1] = f.y;
      }
    }
  } else {
    const T* p = t + (size_t)b * 32 * N + n;
#pragma unroll
    for (int c = 0; c < 32; ++c) v[c] = live ? dh_act_f32(p[(size_t)c * N]) : 0.f;
  }
}

template <bool PM, typename T>
__device__ __forceinline__ void dh_store_pixel(T* __restrict__ t, int b, int n, int N, bool live, const float (&v)[32]) {
  if (!live) return;
  if constexpr (PM && sizeof(T) == 4) {
    float4* p = reinterpret_cast<float4*>(t + ((size_t)b * N + n) * 32);
#pragma unroll
    for (int q = 0; q < 8; ++q) p[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  } else if constexpr (PM) {
    uint4* p = reinterpret_cast<uint4*>(t + ((size_t)b * N + n) * 32);
#pragma unroll
    for (int q = 0; q < 4; ++q)
      p[q] = make_uint4(dh_act_pack2<T>(v[8 * q], v[8 * q + 1]), dh_act_pack2<T>(v[8 * q + 2], v[8 * q + 3]),
                        dh_act_pack2<T>(v[8 * q + 4], v[8 * q + 5]), dh_act_pack2<T>(v[8 * q + 6], v[8 * q + 7]));
  } else {
    T* p = t + (size_t)b * 32 * N + n;
#pragma unroll
    for (int c = 0; c < 32; ++c) p[(size_t)c * N] = dh_act_from<T>(v[c]);
  }
}

// host side: bytes per element of a DH_ACT_* storage type (0: unknown type)
static inline int dh_act_bytes(int act_dtype) {
  return act_dtype == DH_ACT_F32 ? 4 : (act_dtype == DH_ACT_F16 || act_dtype == DH_ACT_BF16) ? 2 : 0;
}
static inline bool dh_aligned(const void* p, int bytes) { return (reinterpret_cast<uintptr_t>(p) & (uintptr_t)(bytes - 1)) == 0; }

// call f(T{}) with T the storage type of act_dtype (validated by the caller with dh_act_bytes)
template <typename F>
static inline int dh_act_dispatch(int act_dtype, F&& f) {
  if (act_dtype == DH_ACT_F16) return f(__half{});
  if (act_dtype == DH_ACT_BF16) return f(__nv_bfloat16{});
  return f(float{});
}
