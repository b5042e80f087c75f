// dahitra_b200 — semantic tokenizer for the TRAINING step: forward (online-softmax partials + merge) and hand-written backward.
//
// Replaces, on the training route, reference models/networks.py:1273-1280 (_forward_semantic_tokens) and what autograd derives
// from it:   a[l][n] = sum_c Wt[l][c] x[c][n];   p = softmax over the N pixels of one image;   tok[l][c] = sum_n p[l][n] x[c][n]
// (x = the post-ReLU squeeze output, 32 channels; 4 tokens).  The backward needs ONE pass over x, because the softmax's
// normalisation term collapses onto the tokens:  sum_n p[l][n] dp[l][n] = sum_c dtok[l][c] tok[l][c]:
//     dp[l][n] = sum_c dtok[l][c] x[c][n]            da[l][n] = p[l][n] (dp[l][n] - sum_c dtok[l][c] tok[l][c])
//     dx[c][n] = sum_l p[l][n] dtok[l][c] + Wt[l][c] da[l][n]          dWt[l][c] = sum_{b, n} da[l][n] x[c][n]
// Layouts: x / dx channel-planar [B][32][N] (NCHW) or pixel-major [B][N][32] (channels_last), stored as fp32, fp16 or bf16
// (train_act.cuh), as in train_decoder.cu; tokens, stats, Wt and every partial are fp32.
// One pixel per thread, 256 pixels per CTA; per-CTA partial sums are written (never accumulated atomically) and reduced by a
// second tiny kernel (forward) or by the caller (dWt): deterministic.
#include "common.cuh"
#include "train_act.cuh"

namespace {

constexpr int TT = 256;          // pixels (= threads) per CTA
constexpr int TP = TT + 4;       // row pitch of the staged [component][pixel] arrays

__device__ __forceinline__ float block_max(float v, float* red) {   // red: >= 8 floats; all threads get the result
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = red[0];
#pragma unroll
  for (int i = 1; i < TT / 32; ++i) r = fmaxf(r, red[i]);
  return r;
}

// per 256-pixel chunk: m[l] = max a, s[l] = sum exp(a - m), t[l][c] = sum exp(a - m) x[c]   -> part[b][chunk][l][34]
template <bool PM, typename TA>
__global__ void __launch_bounds__(TT) tok_fwd_partial_kernel(const TA* __restrict__ x, const float* __restrict__ wt,
                                                             float* __restrict__ part, int N) {
  __shared__ __align__(16) float s_x[32 * TP];
  __shared__ __align__(16) float s_e[4 * TP];
  __shared__ float s_w[128], s_red[8], s_m[4];
  const int b = blockIdx.y, tid = threadIdx.x, n = blockIdx.x * TT + tid;
  const bool live = n < N;
  if (tid < 128) s_w[tid] = wt[tid];
  float v[32];
  dh_load_pixel<PM>(x, b, n, N, live, v);
#pragma unroll
  for (int c = 0; c < 32; ++c) s_x[c * TP + tid] = v[c];
  __syncthreads();
  float a[4];
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    float acc = 0.f;
#pragma unroll
    for (int c = 0; c < 32; ++c) acc = fmaf(s_w[l * 32 + c], v[c], acc);
    a[l] = live ? acc : -INFINITY;
  }
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    const float m = block_max(a[l], s_red);
    if (tid == 0) s_m[l] = m;
    s_e[l * TP + tid] = live ? expf(a[l] - m) : 0.f;
  }
  __syncthreads();
  if (tid < 128) {                                   // thread (l, c): t[l][c]; c == 0 also sums s[l]
    const int l = tid >> 5, c = tid & 31;
    float t = 0.f, s = 0.f;
    const float4* e4 = reinterpret_cast<const float4*>(s_e + l * TP);
    const float4* x4 = reinterpret_cast<const float4*>(s_x + c * TP);
#pragma unroll 4
    for (int p = 0; p < TT / 4; ++p) {
      const float4 e = e4[p], xv = x4[p];
      t = fmaf(e.x, xv.x, t); t = fmaf(e.y, xv.y, t); t = fmaf(e.z, xv.z, t); t = fmaf(e.w, xv.w, t);
      s += (e.x + e.y) + (e.z + e.w);
    }
    float* o = part + (((size_t)b * gridDim.x + blockIdx.x) * 4 + l) * 34;
    o[2 + c] = t;
    if (c == 0) { o[0] = s_m[l]; o[1] = s; }
  }
}

// merge the chunks of one image: tok[b][l][c], stats[b][l] = {M, Z}
__global__ void __launch_bounds__(128) tok_merge_kernel(const float* __restrict__ part, int nchunk, float* __restrict__ tok,
                                                        float* __restrict__ stats) {
  const int b = blockIdx.x, l = threadIdx.x >> 5, c = threadIdx.x & 31;
  const float* p = part + ((size_t)b * nchunk * 4 + l) * 34;
  float M = -INFINITY;
  for (int k = 0; k < nchunk; ++k) M = fmaxf(M, p[(size_t)k * 4 * 34]);
  float Z = 0.f, t = 0.f;
  for (int k = 0; k < nchunk; ++k) {
    const float* q = p + (size_t)k * 4 * 34;
    const float f = expf(q[0] - M);
    Z = fmaf(q[1], f, Z);
    t = fmaf(q[2 + c], f, t);
  }
  tok[((size_t)b * 4 + l) * 32 + c] = t / Z;
  if (c == 0) { stats[(b * 4 + l) * 2] = M; stats[(b * 4 + l) * 2 + 1] = Z; }
}

template <bool PM, typename TA>
__global__ void __launch_bounds__(TT) tok_bwd_kernel(const TA* __restrict__ x, const float* __restrict__ wt,
                                                     const float* __restrict__ tok, const float* __restrict__ stats,
                                                     const float* __restrict__ dtok, TA* __restrict__ dx,
                                                     float* __restrict__ dwt_part, int N) {
  __shared__ __align__(16) float s_x[32 * TP];
  __shared__ __align__(16) float s_da[4 * TP];
  __shared__ float s_w[128], s_dt[128], s_s[4];
  const int b = blockIdx.y, tid = threadIdx.x, n = blockIdx.x * TT + tid;
  const bool live = n < N;
  if (tid < 128) {
    s_w[tid] = wt[tid];
    const float d = dtok[(size_t)b * 128 + tid];
    s_dt[tid] = d;
    const float s = warp_sum(d * tok[(size_t)b * 128 + tid]);       // warp l of the first four: sum_c dtok[l][c] tok[l][c]
    if ((tid & 31) == 0) s_s[tid >> 5] = s;
  }
  float v[32];
  dh_load_pixel<PM>(x, b, n, N, live, v);
#pragma unroll
  for (int c = 0; c < 32; ++c) s_x[c * TP + tid] = v[c];
  __syncthreads();
  float p[4], da[4];
#pragma unroll
  for (int l = 0; l < 4; ++l) {
    float a = 0.f, dp = 0.f;
#pragma unroll
    for (int c = 0; c < 32; ++c) { a = fmaf(s_w[l * 32 + c], v[c], a); dp = fmaf(s_dt[l * 32 + c], v[c], dp); }
    p[l] = live ? expf(a - stats[(b * 4 + l) * 2]) / stats[(b * 4 + l) * 2 + 1] : 0.f;
    da[l] = p[l] * (dp - s_s[l]);
    s_da[l * TP + tid] = da[l];
  }
  if (live) {
    float g[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      float acc = 0.f;
#pragma unroll
      for (int l = 0; l < 4; ++l) acc = fmaf(p[l], s_dt[l * 32 + c], fmaf(s_w[l * 32 + c], da[l], acc));
      g[c] = acc;
    }
    dh_store_pixel<PM>(dx, b, n, N, true, g);
  }
  __syncthreads();
  if (tid < 128) {                                   // dWt partial of this chunk: thread (l, c)
    const int l = tid >> 5, c = tid & 31;
    float t = 0.f;
    const float4* d4 = reinterpret_cast<const float4*>(s_da + l * TP);
    const float4* x4 = reinterpret_cast<const float4*>(s_x + c * TP);
#pragma unroll 4
    for (int q = 0; q < TT / 4; ++q) {
      const float4 d = d4[q], xv = x4[q];
      t = fmaf(d.x, xv.x, t); t = fmaf(d.y, xv.y, t); t = fmaf(d.z, xv.z, t); t = fmaf(d.w, xv.w, t);
    }
    dwt_part[((size_t)b * gridDim.x + blockIdx.x) * 128 + tid] = t;
  }
}

}  // namespace

extern "C" int dahitra_tokenizer_train_chunks(int npix) { return npix > 0 ? dh_cdiv(npix, TT) : 0; }

extern "C" int dahitra_tokenizer_train_fwd_ex(const void* x, const float* w_tok, float* partials, float* tokens, float* stats,
                                              int nimg, int npix, int pixel_major, int act_dtype, void* stream) {
  const int eb = dh_act_bytes(act_dtype);
  DH_REQUIRE(eb > 0, DH_E_VARIANT);
  DH_REQUIRE(x && w_tok && partials && tokens && stats, DH_E_NULL);
  DH_REQUIRE(nimg > 0 && npix > 0 && nimg <= 65535, DH_E_SHAPE);
  DH_REQUIRE(dh_aligned(x, pixel_major ? 16 : eb), DH_E_ALIGN);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const dim3 grid(dh_cdiv(npix, TT), nimg);
  dh_act_dispatch(act_dtype, [&](auto t) {
    using TA = decltype(t);
    if (pixel_major) tok_fwd_partial_kernel<true, TA><<<grid, TT, 0, s>>>(static_cast<const TA*>(x), w_tok, partials, npix);
    else tok_fwd_partial_kernel<false, TA><<<grid, TT, 0, s>>>(static_cast<const TA*>(x), w_tok, partials, npix);
    return 0;
  });
  DH_CHECK_LAUNCH();
  tok_merge_kernel<<<nimg, 128, 0, s>>>(partials, (int)grid.x, tokens, stats);
  DH_CHECK_LAUNCH();
  return 0;
}

extern "C" int dahitra_tokenizer_train_bwd_ex(const void* x, const float* w_tok, const float* tokens, const float* stats,
                                              const float* dtokens, void* dx, float* dw_partial, int nimg, int npix,
                                              int pixel_major, int act_dtype, void* stream) {
  const int eb = dh_act_bytes(act_dtype);
  DH_REQUIRE(eb > 0, DH_E_VARIANT);
  DH_REQUIRE(x && w_tok && tokens && stats && dtokens && dx && dw_partial, DH_E_NULL);
  DH_REQUIRE(nimg > 0 && npix > 0 && nimg <= 65535, DH_E_SHAPE);
  DH_REQUIRE(dh_aligned(x, pixel_major ? 16 : eb) && dh_aligned(dx, pixel_major ? 16 : eb), DH_E_ALIGN);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const dim3 grid(dh_cdiv(npix, TT), nimg);
  dh_act_dispatch(act_dtype, [&](auto t) {
    using TA = decltype(t);
    const TA* xa = static_cast<const TA*>(x);
    TA* da = static_cast<TA*>(dx);
    if (pixel_major) tok_bwd_kernel<true, TA><<<grid, TT, 0, s>>>(xa, w_tok, tokens, stats, dtokens, da, dw_partial, npix);
    else tok_bwd_kernel<false, TA><<<grid, TT, 0, s>>>(xa, w_tok, tokens, stats, dtokens, da, dw_partial, npix);
    return 0;
  });
  DH_CHECK_LAUNCH();
  return 0;
}

extern "C" int dahitra_tokenizer_train_fwd(const float* x, const float* w_tok, float* partials, float* tokens, float* stats,
                                           int nimg, int npix, int pixel_major, void* stream) {
  return dahitra_tokenizer_train_fwd_ex(x, w_tok, partials, tokens, stats, nimg, npix, pixel_major, DH_ACT_F32, stream);
}

extern "C" int dahitra_tokenizer_train_bwd(const float* x, const float* w_tok, const float* tokens, const float* stats,
                                           const float* dtokens, float* dx, float* dw_partial, int nimg, int npix,
                                           int pixel_major, void* stream) {
  return dahitra_tokenizer_train_bwd_ex(x, w_tok, tokens, stats, dtokens, dx, dw_partial, nimg, npix, pixel_major, DH_ACT_F32,
                                        stream);
}
