// dahitra_b200 — helpers for the split16 activation format of conv_tc3.cu (hi = f16(a), lo = f16(2^11 (a - hi)); two
// FP16 planes of the tensor's shape, the lo plane `n` elements after the hi plane):
//   * fp32 <-> split16 conversion (block tests, and the boundary of code that keeps fp32 tensors),
//   * MaxPool2d(3, 2, 1) on a split16 NHWC tensor (reference models/networks.py:1123,1128 — the same module applied after the
//     stem and after layer2): the order of the values is the lexicographic order of their (hi, lo) pairs, so the pool runs
//     on packed halves and copies the winner's planes;
//   * the same pool on ONE FP16 plane (the h16 mode): a max of 16-bit values, exact.
#include "tc_common.cuh"
#include <cuda_fp16.h>

using namespace dhtc;

namespace {

__device__ __forceinline__ void sp_split8(const float (&v)[8], uint4& hi, uint4& lo) {
  hi.x = pack_f16x2_sat(v[0], v[1]); hi.y = pack_f16x2_sat(v[2], v[3]); hi.z = pack_f16x2_sat(v[4], v[5]); hi.w = pack_f16x2_sat(v[6], v[7]);
  lo.x = pack_f16x2_sat((v[0] - f16_lo(hi.x)) * 2048.f, (v[1] - f16_hi(hi.x)) * 2048.f);
  lo.y = pack_f16x2_sat((v[2] - f16_lo(hi.y)) * 2048.f, (v[3] - f16_hi(hi.y)) * 2048.f);
  lo.z = pack_f16x2_sat((v[4] - f16_lo(hi.z)) * 2048.f, (v[5] - f16_hi(hi.z)) * 2048.f);
  lo.w = pack_f16x2_sat((v[6] - f16_lo(hi.w)) * 2048.f, (v[7] - f16_hi(hi.w)) * 2048.f);
}
__device__ __forceinline__ void sp_join8(uint4 hi, uint4 lo, float (&v)[8]) {
  constexpr float S = 1.0f / 2048.0f;
  v[0] = fmaf(f16_lo(lo.x), S, f16_lo(hi.x)); v[1] = fmaf(f16_hi(lo.x), S, f16_hi(hi.x));
  v[2] = fmaf(f16_lo(lo.y), S, f16_lo(hi.y)); v[3] = fmaf(f16_hi(lo.y), S, f16_hi(hi.y));
  v[4] = fmaf(f16_lo(lo.z), S, f16_lo(hi.z)); v[5] = fmaf(f16_hi(lo.z), S, f16_hi(hi.z));
  v[6] = fmaf(f16_lo(lo.w), S, f16_lo(hi.w)); v[7] = fmaf(f16_hi(lo.w), S, f16_hi(hi.w));
}

__global__ void __launch_bounds__(256) split_pack_kernel(const float* __restrict__ in, size_t n8, size_t n, uint16_t* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
    const float4 a = ldg4(in + i * 8), b = ldg4(in + i * 8 + 4);
    const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint4 hi, lo;
    sp_split8(v, hi, lo);
    *reinterpret_cast<uint4*>(out + i * 8) = hi;
    *reinterpret_cast<uint4*>(out + n + i * 8) = lo;
  }
}
__global__ void __launch_bounds__(256) split_unpack_kernel(const uint16_t* __restrict__ in, size_t n8, size_t n, float* __restrict__ out) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
    const uint4 hi = __ldg(reinterpret_cast<const uint4*>(in + i * 8)), lo = __ldg(reinterpret_cast<const uint4*>(in + n + i * 8));
    float v[8];
    sp_join8(hi, lo, v);
    st4(out + i * 8, make_float4(v[0], v[1], v[2], v[3]));
    st4(out + i * 8 + 4, make_float4(v[4], v[5], v[6], v[7]));
  }
}

// lexicographic max on (hi, lo) pairs of packed halves: a > b  <=>  hi_a > hi_b, or hi_a == hi_b and lo_a > lo_b (|lo| / 2048 never
// exceeds half an ulp of hi), so the pool needs no conversion to fp32 and no re-split: 7 packed instructions per two elements
__device__ __forceinline__ void lexmax2(uint32_t& mh, uint32_t& ml, uint32_t h, uint32_t l) {
  const __half2 a = *reinterpret_cast<const __half2*>(&h), m = *reinterpret_cast<const __half2*>(&mh);
  const uint32_t gt = __hgt2_mask(a, m), eq = __heq2_mask(a, m);
  const __half2 lm = __hmax2(*reinterpret_cast<const __half2*>(&l), *reinterpret_cast<const __half2*>(&ml));
  ml = (gt & l) | (eq & *reinterpret_cast<const uint32_t*>(&lm)) | (~(gt | eq) & ml);
  mh = (gt & h) | (~gt & mh);
}

// one thread = 8 channels of one output pixel (16-byte loads / stores per plane)
__global__ void __launch_bounds__(256)
maxpool_split_kernel(const uint16_t* __restrict__ in, int N, int H, int W, int C, uint16_t* __restrict__ out) {
  const int OH = H / 2, OW = W / 2, C8 = C / 8;
  const size_t total = (size_t)N * OH * OW * C8, plane_in = (size_t)N * H * W * C, plane_out = (size_t)N * OH * OW * C;
  pdl_wait();
  pdl_launch_dependents();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c8 = (int)(i % C8);
  size_t p = i / C8;
  const int ox = (int)(p % OW); p /= OW;
  const int oy = (int)(p % OH);
  const int n = (int)(p / OH);
  uint4 mh = make_uint4(0xFC00FC00u, 0xFC00FC00u, 0xFC00FC00u, 0xFC00FC00u), ml = mh;      // -inf
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    const int iy = 2 * oy + dy;
    if (iy < 0 || iy >= H) continue;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int ix = 2 * ox + dx;
      if (ix < 0 || ix >= W) continue;
      const size_t o = (((size_t)n * H + iy) * W + ix) * C + c8 * 8;
      const uint4 hi = __ldg(reinterpret_cast<const uint4*>(in + o)), lo = __ldg(reinterpret_cast<const uint4*>(in + plane_in + o));
      lexmax2(mh.x, ml.x, hi.x, lo.x); lexmax2(mh.y, ml.y, hi.y, lo.y); lexmax2(mh.z, ml.z, hi.z, lo.z); lexmax2(mh.w, ml.w, hi.w, lo.w);
    }
  }
  const size_t o = (((size_t)n * OH + oy) * OW + ox) * C + c8 * 8;
  *reinterpret_cast<uint4*>(out + o) = mh;
  *reinterpret_cast<uint4*>(out + plane_out + o) = ml;
}

// one thread = 8 channels of one output pixel (16-byte loads / stores)
__global__ void __launch_bounds__(256)
maxpool_h16_kernel(const uint16_t* __restrict__ in, int N, int H, int W, int C, uint16_t* __restrict__ out) {
  const int OH = H / 2, OW = W / 2, C8 = C / 8;
  const size_t total = (size_t)N * OH * OW * C8;
  pdl_wait();
  pdl_launch_dependents();
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c8 = (int)(i % C8);
  size_t p = i / C8;
  const int ox = (int)(p % OW); p /= OW;
  const int oy = (int)(p % OH);
  const int n = (int)(p / OH);
  __half2 m[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) m[k] = __half2half2(__ushort_as_half((unsigned short)0xFC00u));    // -inf
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    const int iy = 2 * oy + dy;
    if (iy < 0 || iy >= H) continue;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int ix = 2 * ox + dx;
      if (ix < 0 || ix >= W) continue;
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(in + (((size_t)n * H + iy) * W + ix) * C + c8 * 8));
      const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
      for (int k = 0; k < 4; ++k) m[k] = __hmax2(m[k], h[k]);
    }
  }
  *reinterpret_cast<uint4*>(out + (((size_t)n * OH + oy) * OW + ox) * C + c8 * 8) = *reinterpret_cast<const uint4*>(m);
}

int grid_for(size_t items) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const size_t want = (items + 255) / 256, cap = (size_t)sms * 8;
  return (int)(want < cap ? (want ? want : 1) : cap);
}
}  // namespace

int dh_launch_split_pack(const float* in, size_t n, void* out, cudaStream_t s) {
  DH_REQUIRE(in && out, DH_E_NULL);
  DH_REQUIRE(n % 8 == 0 && n > 0, DH_E_SHAPE);
  DH_REQUIRE(dh_aligned16(in) && dh_aligned16(out), DH_E_ALIGN);
  split_pack_kernel<<<grid_for(n / 8), 256, 0, s>>>(in, n / 8, n, reinterpret_cast<uint16_t*>(out));
  DH_CHECK_LAUNCH();
  return 0;
}
int dh_launch_split_unpack(const void* in, size_t n, float* out, cudaStream_t s) {
  DH_REQUIRE(in && out, DH_E_NULL);
  DH_REQUIRE(n % 8 == 0 && n > 0, DH_E_SHAPE);
  DH_REQUIRE(dh_aligned16(in) && dh_aligned16(out), DH_E_ALIGN);
  split_unpack_kernel<<<grid_for(n / 8), 256, 0, s>>>(reinterpret_cast<const uint16_t*>(in), n / 8, n, out);
  DH_CHECK_LAUNCH();
  return 0;
}
int dh_launch_maxpool_split(const void* in, int N, int H, int W, int C, void* out, cudaStream_t s) {
  DH_REQUIRE(in && out, DH_E_NULL);
  DH_REQUIRE(N > 0 && H >= 2 && W >= 2 && H % 2 == 0 && W % 2 == 0 && C % 8 == 0, DH_E_SHAPE);
  DH_REQUIRE(dh_aligned16(in) && dh_aligned16(out), DH_E_ALIGN);
  const size_t items = (size_t)N * (H / 2) * (W / 2) * (C / 8);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)((items + 255) / 256)); cfg.blockDim = dim3(256); cfg.stream = s;
  cudaLaunchAttribute at[1];
  cfg.attrs = at; cfg.numAttrs = dh_pdl_attr(at);
  const cudaError_t e = cudaLaunchKernelEx(&cfg, maxpool_split_kernel, reinterpret_cast<const uint16_t*>(in), N, H, W, C,
                                           reinterpret_cast<uint16_t*>(out));
  if (e != cudaSuccess) return (int)e;
  DH_CHECK_LAUNCH();
  return 0;
}
int dh_launch_maxpool_h16(const void* in, int N, int H, int W, int C, void* out, cudaStream_t s) {
  DH_REQUIRE(in && out, DH_E_NULL);
  DH_REQUIRE(N > 0 && H >= 2 && W >= 2 && H % 2 == 0 && W % 2 == 0 && C % 8 == 0, DH_E_SHAPE);
  DH_REQUIRE(dh_aligned16(in) && dh_aligned16(out), DH_E_ALIGN);
  const size_t items = (size_t)N * (H / 2) * (W / 2) * (C / 8);
  return dh_launch(maxpool_h16_kernel, dim3((unsigned)((items + 255) / 256)), dim3(256), 0, s,
                   reinterpret_cast<const uint16_t*>(in), N, H, W, C, reinterpret_cast<uint16_t*>(out));
}
