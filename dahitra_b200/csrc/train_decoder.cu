// dahitra_b200 — pixel decoder for the TRAINING step: forward that keeps the layer inputs, and the hand-written backward.
//
// Replaces, on the training route, the per-pixel part of reference models/help_funcs.py:66-114,170-186 (TransformerDecoder:
// depth x [Residual2(PreNorm2(Cross_Attention)), Residual(PreNorm(FeedForward))]) and everything autograd derives from it.
// The arithmetic is the collapsed algebra of the inference kernel (DESIGN.md "pixel_decoder"), in plain fp32 FMAs: the 4
// memory tokens are constant over the pixels, so per (image, layer) the q / k / v / out projections fold into two small
// matrices that the HOST builds with differentiable torch ops (modules.PixelDecoder.train_tables):
//     xn = LN0(x)                        (normalisation only; the LayerNorm affine is folded into A / W1)
//     d  = c0 + xn A          A [32][K]  K = 4 * heads,  k = head * 4 + token
//     p  = softmax over each head's 4 entries of d
//     y  = x + bo + p Bv      Bv[K][32]
//     yn = LN0(y)
//     h  = b1 + yn W1         W1[32][32] (input-major)
//     z  = y + b2 + gelu(h) W2           W2[32][32] (input-major)
// The backward kernel returns dL/dx and the gradient of EVERY table entry (summed over the CTA's pixels; the host adds the
// per-CTA partials, a deterministic two-level reduction), and autograd carries the table gradients back to Wq, Wk, Wv, Wo, the
// LayerNorm parameters, the MLP weights and — through the tokens — the tokenizer, the token encoder and the trunk.
//
// Layout: x, out, dx, dout are channel-planar [B][32][N] (= the NCHW tensors of the reference, flattened over h, w): one thread
// per pixel reads and writes fully coalesced rows, and no transpose to (B, N, 32) is ever made; or pixel-major [B][N][32]
// (channels_last).  Their storage type TA is fp32, fp16 or bf16 (train_act.cuh: what autocast hands over); the saved layer
// inputs xs stay fp32, so the backward recomputes exactly what the forward computed.
// Table [B][L][DH_TRAIN_TAB_FLOATS(K)]:  A 32K | c0 K | Bv 32K | bo 32 | W1 1024 | b1 32 | W2 1024 | b2 32.
//
// Kernel structure: 128 pixels per CTA, one pixel per thread.  Every per-pixel vector that feeds a contraction lives in shared
// memory as [component][pixel] (row pitch 132 floats: conflict-free both for the per-thread column accesses and for the 16-byte
// row reads of the weight-gradient pass); contractions keep their outputs in registers and read the weights as warp-uniform
// 16-byte broadcasts.  The weight gradients are the third kind of product: out[i][j] = sum over the CTA's pixels of a[i][p] b[j][p],
// each thread owning 4-8 entries.  Products issue as packed FFMA2 on the register pairs of the 128-bit loads.
// Bound (ncu, profiles/r02_ncu_full_decoder_train_bwd_level3.txt): the shared-memory pipe (74 %; FMA pipe 41 %) — one 16-byte
// weight read per four FMAs.  Tried and not kept: two pixels per thread (64-thread CTAs; each weight read feeds two pixels,
// 1.8x fewer shared-memory wavefronts): correct, but 255 registers with spills and four warps per SM made the backward 40 %
// SLOWER (0.67 -> 0.86 ms at level 3) — the kernel needs its eight warps per SM to cover the shared-memory latency.
#include "common.cuh"
#include "train_act.cuh"

namespace {

// packed fp32 pairs (sm_100 FFMA2: two IEEE fp32 FMAs per issued instruction, lane-wise identical to scalar FMAs).  Every
// contraction below keeps its sums as register pairs so that the products of one 128-bit weight / vector load issue as FFMA2.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  unsigned long long ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  float2 d;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(rd));
  return d;
}

constexpr int PT = 128;        // pixels (= threads) per CTA
constexpr int PITCH = PT + 4;  // floats per row of a staged vector
constexpr float LN_EPS = 1e-5f;

struct TabOff {
  int A, c0, Bv, bo, W1, b1, W2, b2, T;
};
__host__ __device__ constexpr TabOff tab_off(int K) {
  return TabOff{0, 32 * K, 33 * K, 65 * K, 65 * K + 32, 65 * K + 32 + 1024, 65 * K + 64 + 1024, 65 * K + 64 + 2048, 65 * K + 96 + 2048};
}

// acc[k] += sum_c in[c][tid] * W[c][k]      (W input-major [CIN][KOUT] in shared memory, warp-uniform reads)
template <int CIN, int KOUT>
__device__ __forceinline__ void matvec(const float* __restrict__ in_col, const float* __restrict__ W, float (&acc)[KOUT]) {
  float2 a2[KOUT / 2];
#pragma unroll
  for (int k = 0; k < KOUT / 2; ++k) a2[k] = make_float2(acc[2 * k], acc[2 * k + 1]);
#pragma unroll 4
  for (int c = 0; c < CIN; ++c) {
    const float v = in_col[c * PITCH];
    const float2 vv = make_float2(v, v);
    const float4* w4 = reinterpret_cast<const float4*>(W + c * KOUT);
#pragma unroll
    for (int q = 0; q < KOUT / 4; ++q) {
      const float4 w = w4[q];
      a2[2 * q] = ffma2(vv, make_float2(w.x, w.y), a2[2 * q]);
      a2[2 * q + 1] = ffma2(vv, make_float2(w.z, w.w), a2[2 * q + 1]);
    }
  }
#pragma unroll
  for (int k = 0; k < KOUT / 2; ++k) { acc[2 * k] = a2[k].x; acc[2 * k + 1] = a2[k].y; }
}

// out[j][tid] = sum_c W[j][c] * in[c]       (rows of the same input-major matrix dotted with a register vector: the transposed
// product of the backward pass; eight rows at a time for independent FMA chains)
template <int CIN, int JOUT>
__device__ __forceinline__ void matvec_t(const float (&in)[CIN], const float* __restrict__ W, float* __restrict__ out_col) {
#pragma unroll 1
  for (int j = 0; j < JOUT; j += 8) {
    float2 a[8];                                   // (sum over even, sum over odd input components) of eight rows
#pragma unroll
    for (int r = 0; r < 8; ++r) a[r] = make_float2(0.f, 0.f);
#pragma unroll
    for (int q = 0; q < CIN / 4; ++q) {
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        const float4 w = reinterpret_cast<const float4*>(W + (j + r) * CIN)[q];
        a[r] = ffma2(make_float2(w.x, w.y), make_float2(in[4 * q], in[4 * q + 1]), a[r]);
        a[r] = ffma2(make_float2(w.z, w.w), make_float2(in[4 * q + 2], in[4 * q + 3]), a[r]);
      }
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) out_col[(j + r) * PITCH] = a[r].x + a[r].y;
  }
}

template <int C>
__device__ __forceinline__ void load_col(const float* __restrict__ col, float (&v)[C]) {
#pragma unroll
  for (int c = 0; c < C; ++c) v[c] = col[c * PITCH];
}
template <int C>
__device__ __forceinline__ void store_col(float* __restrict__ col, const float (&v)[C]) {
#pragma unroll
  for (int c = 0; c < C; ++c) col[c * PITCH] = v[c];
}

// LayerNorm without affine over the 32 channels (biased variance, eps 1e-5: nn.LayerNorm(32))
__device__ __forceinline__ float layer_norm32(const float (&x)[32], float (&xn)[32]) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < 32; ++c) s += x[c];
  const float mean = s * (1.f / 32.f);
  float q = 0.f;
#pragma unroll
  for (int c = 0; c < 32; ++c) { const float d = x[c] - mean; q = fmaf(d, d, q); }
  const float rstd = 1.f / sqrtf(q * (1.f / 32.f) + LN_EPS);
#pragma unroll
  for (int c = 0; c < 32; ++c) xn[c] = (x[c] - mean) * rstd;
  return rstd;
}
// dx = rstd * (dxn - mean(dxn) - xn * mean(dxn * xn))
__device__ __forceinline__ void layer_norm32_bwd(const float (&dxn)[32], const float (&xn)[32], float rstd, float (&dx)[32]) {
  float s = 0.f, t = 0.f;
#pragma unroll
  for (int c = 0; c < 32; ++c) { s += dxn[c]; t = fmaf(dxn[c], xn[c], t); }
  s *= (1.f / 32.f); t *= (1.f / 32.f);
#pragma unroll
  for (int c = 0; c < 32; ++c) dx[c] = rstd * (dxn[c] - s - xn[c] * t);
}

template <int K>
__device__ __forceinline__ void softmax4(float (&d)[K]) {
#pragma unroll
  for (int h = 0; h < K / 4; ++h) {
    const float m = fmaxf(fmaxf(d[4 * h], d[4 * h + 1]), fmaxf(d[4 * h + 2], d[4 * h + 3]));
    const float e0 = expf(d[4 * h] - m), e1 = expf(d[4 * h + 1] - m), e2 = expf(d[4 * h + 2] - m), e3 = expf(d[4 * h + 3] - m);
    const float inv = 1.f / (e0 + e1 + e2 + e3);
    d[4 * h] = e0 * inv; d[4 * h + 1] = e1 * inv; d[4 * h + 2] = e2 * inv; d[4 * h + 3] = e3 * inv;
  }
}

__device__ __forceinline__ void load_table(const float* __restrict__ g, float* __restrict__ s, int T) {
  for (int i = threadIdx.x * 4; i < T; i += PT * 4) *reinterpret_cast<float4*>(s + i) = __ldg(reinterpret_cast<const float4*>(g + i));
}

// ------------------------------------------------------------------------------------------------ forward (training)
template <int K, bool PM, typename TA>
__global__ void __launch_bounds__(PT) decoder_train_fwd_kernel(const TA* __restrict__ x, const float* __restrict__ table,
                                                               float* __restrict__ xs, TA* __restrict__ out, int B, int N, int L) {
  constexpr TabOff O = tab_off(K);
  extern __shared__ __align__(16) float smem[];
  float* tab = smem;                       // O.T floats
  float* bufA = smem + O.T;                // [32][PITCH]
  float* bufB = bufA + 32 * PITCH;         // [32][PITCH]
  const int b = blockIdx.y, tid = threadIdx.x, n = blockIdx.x * PT + tid;
  const bool live = n < N;
  float v[32];
  dh_load_pixel<PM>(x, b, n, N, live, v);
  for (int l = 0; l < L; ++l) {
    __syncthreads();                                                   // the previous layer is done with the table
    load_table(table + ((size_t)b * L + l) * O.T, tab, O.T);
    dh_store_pixel<false>(xs + (size_t)l * B * 32 * N, b, n, N, live, v);  // layer inputs are kept planar (coalesced both ways)
    {
      float xn[32];
      layer_norm32(v, xn);
      store_col(bufA + tid, xn);
    }
    __syncthreads();                                                   // table loaded (own column needs no barrier)
    {
      float d[K];
#pragma unroll
      for (int k = 0; k < K; ++k) d[k] = tab[O.c0 + k];
      matvec<32, K>(bufA + tid, tab + O.A, d);
      softmax4<K>(d);
      store_col(bufB + tid, d);
    }
#pragma unroll
    for (int c = 0; c < 32; ++c) v[c] += tab[O.bo + c];
    matvec<K, 32>(bufB + tid, tab + O.Bv, v);                          // y = x + bo + p Bv
    {
      float yn[32];
      layer_norm32(v, yn);
      store_col(bufA + tid, yn);
    }
    {
      float h[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) h[j] = tab[O.b1 + j];
      matvec<32, 32>(bufA + tid, tab + O.W1, h);
#pragma unroll
      for (int j = 0; j < 32; ++j) h[j] = gelu_erf(h[j]);
      store_col(bufB + tid, h);
    }
#pragma unroll
    for (int c = 0; c < 32; ++c) v[c] += tab[O.b2 + c];
    matvec<32, 32>(bufB + tid, tab + O.W2, v);                         // z = y + b2 + gelu(h) W2
  }
  dh_store_pixel<PM>(out, b, n, N, live, v);
}

// ------------------------------------------------------------------------------------------------ backward
// out[i][j] = sum_p a[i][p] b[j][p] over the CTA's 128 pixels, written (not accumulated) to g_w[i * J + j]; g_bias[j] = sum_p b[j][p]
template <int I, int J>
__device__ __forceinline__ void wgrad(const float* __restrict__ a, const float* __restrict__ bm, float* __restrict__ g_w,
                                      float* __restrict__ g_bias) {
  constexpr int TPR = PT / I;            // threads per row of the result
  constexpr int M = J / TPR;             // entries per thread
  const int i = threadIdx.x / TPR, j0 = threadIdx.x % TPR;
  float2 acc[M];                                   // (sum over even, sum over odd pixels)
  float bsum[M];
#pragma unroll
  for (int m = 0; m < M; ++m) { acc[m] = make_float2(0.f, 0.f); bsum[m] = 0.f; }
  const float4* a4 = reinterpret_cast<const float4*>(a + i * PITCH);
#pragma unroll 2
  for (int p = 0; p < PT / 4; ++p) {
    const float4 av = a4[p];
#pragma unroll
    for (int m = 0; m < M; ++m) {
      const float4 bv = reinterpret_cast<const float4*>(bm + (j0 + TPR * m) * PITCH)[p];
      acc[m] = ffma2(make_float2(av.x, av.y), make_float2(bv.x, bv.y), acc[m]);
      acc[m] = ffma2(make_float2(av.z, av.w), make_float2(bv.z, bv.w), acc[m]);
      if (i == 0) bsum[m] += (bv.x + bv.y) + (bv.z + bv.w);
    }
  }
#pragma unroll
  for (int m = 0; m < M; ++m) {
    g_w[i * J + j0 + TPR * m] = acc[m].x + acc[m].y;
    if (i == 0) g_bias[j0 + TPR * m] = bsum[m];
  }
}

template <int K, bool PM, typename TA>
__global__ void __launch_bounds__(PT, 2) decoder_train_bwd_kernel(const TA* __restrict__ dout, const float* __restrict__ xs,
                                                                  const float* __restrict__ table, TA* __restrict__ dx,
                                                                  float* __restrict__ dtab, int B, int N, int L) {
  constexpr TabOff O = tab_off(K);
  extern __shared__ __align__(16) float smem[];
  // five staged vectors (so that two CTAs fit one SM); xn is recomputed from the layer input where it is needed a second time
  float* tab = smem;
  float* s_p = smem + O.T;                 // [K][PITCH]    softmax probabilities
  float* s_yn = s_p + K * PITCH;           // [32][PITCH]   xn (forward), yn, later xn again (for dA)
  float* s_g = s_yn + 32 * PITCH;          // [32][PITCH]   gelu(h); later dg, dyn, dy, dxn
  float* s_gp = s_g + 32 * PITCH;          // [32][PITCH]   gelu'(h); later dh (in place)
  float* s_dz = s_gp + 32 * PITCH;         // [32][PITCH]   dz; later dp, dd (first K rows)
  const int b = blockIdx.y, tid = threadIdx.x, n = blockIdx.x * PT + tid;
  const bool live = n < N;
  float dz[32];
  dh_load_pixel<PM>(dout, b, n, N, live, dz);
  for (int l = L - 1; l >= 0; --l) {
    __syncthreads();                                                   // the previous layer's last wgrad / table reads are done
    load_table(table + ((size_t)b * L + l) * O.T, tab, O.T);
    float* gt = dtab + (((size_t)b * gridDim.x + blockIdx.x) * L + l) * O.T;     // this CTA's partial of the layer's table gradient
    const float* xl = xs + (size_t)l * B * 32 * N;
    float rstd1, rstd2;
    // ---- recompute the layer's forward; keep p, yn, gelu(h), gelu'(h) in shared memory
    {
      float v[32];
      dh_load_pixel<false>(xl, b, n, N, live, v);
      {
        float xn[32];
        rstd1 = layer_norm32(v, xn);
        store_col(s_yn + tid, xn);
      }
      __syncthreads();                                                 // table loaded
      {
        float d[K];
#pragma unroll
        for (int k = 0; k < K; ++k) d[k] = tab[O.c0 + k];
        matvec<32, K>(s_yn + tid, tab + O.A, d);
        softmax4<K>(d);
        store_col(s_p + tid, d);
      }
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] += tab[O.bo + c];
      matvec<K, 32>(s_p + tid, tab + O.Bv, v);
      {
        float yn[32];
        rstd2 = layer_norm32(v, yn);
        store_col(s_yn + tid, yn);
      }
      float h[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) h[j] = tab[O.b1 + j];
      matvec<32, 32>(s_yn + tid, tab + O.W1, h);
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const float cdf = 0.5f * (1.f + erff(h[j] * 0.70710678118654752440f));
        const float pdf = 0.39894228040143267794f * expf(-0.5f * h[j] * h[j]);
        s_g[j * PITCH + tid] = h[j] * cdf;
        s_gp[j * PITCH + tid] = fmaf(h[j], pdf, cdf);
      }
    }
    // ---- z = y + b2 + g W2 :  dW2[j][c] = sum g[j] dz[c], db2 = sum dz, dg = W2 dz
    store_col(s_dz + tid, dz);
    __syncthreads();                                                   // (1)
    wgrad<32, 32>(s_g, s_dz, gt + O.W2, gt + O.b2);
    __syncthreads();                                                   // (2) s_g is overwritten below
    matvec_t<32, 32>(dz, tab + O.W2, s_g + tid);                       // dg -> s_g (own column)
#pragma unroll
    for (int j = 0; j < 32; ++j) s_gp[j * PITCH + tid] *= s_g[j * PITCH + tid];      // dh = dg * gelu'(h), in place
    __syncthreads();                                                   // (3)
    // ---- h = b1 + yn W1 :  dW1[c][j] = sum yn[c] dh[j], db1 = sum dh, dyn = W1 dh
    wgrad<32, 32>(s_yn, s_gp, gt + O.W1, gt + O.b1);
    {
      float dh[32];
      load_col(s_gp + tid, dh);
      matvec_t<32, 32>(dh, tab + O.W1, s_g + tid);                     // dyn -> s_g (own column; s_g is not read by the wgrad above)
    }
    {
      float dyn[32], yn[32], t[32];
      load_col(s_g + tid, dyn);
      load_col(s_yn + tid, yn);
      layer_norm32_bwd(dyn, yn, rstd2, t);
#pragma unroll
      for (int c = 0; c < 32; ++c) dz[c] += t[c];                      // dy = dz (residual) + LayerNorm backward
    }
    store_col(s_g + tid, dz);                                          // dy staged
    __syncthreads();                                                   // (4) also: the wgrad above has finished reading s_yn / s_gp
    // ---- y = x + bo + p Bv :  dBv[k][c] = sum p[k] dy[c], dbo = sum dy, dp = Bv dy
    wgrad<K, 32>(s_p, s_g, gt + O.Bv, gt + O.bo);
    matvec_t<32, K>(dz, tab + O.Bv, s_dz + tid);                       // dp -> s_dz (own column; last read before barrier (2))
    {
      float v[32], xn[32];                                             // xn again (s_yn is free since barrier (4))
      dh_load_pixel<false>(xl, b, n, N, live, v);
      layer_norm32(v, xn);
      store_col(s_yn + tid, xn);
    }
    {
      float p[K], dp[K];
      load_col(s_p + tid, p);
      load_col(s_dz + tid, dp);
#pragma unroll
      for (int h = 0; h < K / 4; ++h) {
        const float dot = p[4 * h] * dp[4 * h] + p[4 * h + 1] * dp[4 * h + 1] + p[4 * h + 2] * dp[4 * h + 2] + p[4 * h + 3] * dp[4 * h + 3];
#pragma unroll
        for (int j = 0; j < 4; ++j) dp[4 * h + j] = p[4 * h + j] * (dp[4 * h + j] - dot);
      }
      store_col(s_dz + tid, dp);                                       // dd staged
      __syncthreads();                                                 // (5) also: the Bv wgrad has finished reading s_g
      // ---- d = c0 + xn A :  dA[c][k] = sum xn[c] dd[k], dc0 = sum dd, dxn = A dd
      wgrad<32, K>(s_yn, s_dz, gt + O.A, gt + O.c0);
      matvec_t<K, 32>(dp, tab + O.A, s_g + tid);                       // dxn -> s_g (own column; not read by this wgrad)
    }
    {
      float dxn[32], xn[32], t[32];
      load_col(s_g + tid, dxn);
      load_col(s_yn + tid, xn);
      layer_norm32_bwd(dxn, xn, rstd1, t);
#pragma unroll
      for (int c = 0; c < 32; ++c) dz[c] += t[c];                      // dx = dy (residual) + LayerNorm backward
    }
  }
  dh_store_pixel<PM>(dx, b, n, N, live, dz);
}

template <int K, bool PM, typename TA>
int launch_fwd(const TA* x, const float* table, float* xs, TA* out, int B, int N, int L, cudaStream_t s) {
  constexpr TabOff O = tab_off(K);
  const size_t smem = (size_t)(O.T + 2 * 32 * PITCH) * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(decoder_train_fwd_kernel<K, PM, TA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  decoder_train_fwd_kernel<K, PM, TA><<<dim3(dh_cdiv(N, PT), B), PT, smem, s>>>(x, table, xs, out, B, N, L);
  DH_CHECK_LAUNCH();
  return 0;
}
template <int K, bool PM, typename TA>
int launch_bwd(const TA* dout, const float* xs, const float* table, TA* dx, float* dtab, int B, int N, int L, cudaStream_t s) {
  constexpr TabOff O = tab_off(K);
  const size_t smem = (size_t)(O.T + (4 * 32 + K) * PITCH) * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(decoder_train_bwd_kernel<K, PM, TA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  decoder_train_bwd_kernel<K, PM, TA><<<dim3(dh_cdiv(N, PT), B), PT, smem, s>>>(dout, xs, table, dx, dtab, B, N, L);
  DH_CHECK_LAUNCH();
  return 0;
}

}  // namespace

extern "C" int dahitra_pixel_decoder_train_blocks(int npix) { return npix > 0 ? dh_cdiv(npix, PT) : 0; }

extern "C" int dahitra_pixel_decoder_train_fwd_ex(const void* x, const float* tables, float* xs, void* out, int nimg, int npix,
                                                  int heads, int depth, int pixel_major, int act_dtype, void* stream) {
  const int eb = dh_act_bytes(act_dtype);
  DH_REQUIRE(eb > 0, DH_E_VARIANT);
  DH_REQUIRE(x && tables && xs && out, DH_E_NULL);
  DH_REQUIRE(nimg > 0 && npix > 0 && depth > 0 && nimg <= 65535, DH_E_SHAPE);
  DH_REQUIRE(heads == 4 || heads == 8, DH_E_SHAPE);
  const int xal = pixel_major ? 16 : eb;
  DH_REQUIRE(dh_aligned16(tables) && dh_aligned(x, xal) && dh_aligned(out, xal), DH_E_ALIGN);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return dh_act_dispatch(act_dtype, [&](auto t) {
    using TA = decltype(t);
    const TA* xa = static_cast<const TA*>(x);
    TA* oa = static_cast<TA*>(out);
    if (pixel_major)
      return heads == 4 ? launch_fwd<16, true>(xa, tables, xs, oa, nimg, npix, depth, s) : launch_fwd<32, true>(xa, tables, xs, oa, nimg, npix, depth, s);
    return heads == 4 ? launch_fwd<16, false>(xa, tables, xs, oa, nimg, npix, depth, s) : launch_fwd<32, false>(xa, tables, xs, oa, nimg, npix, depth, s);
  });
}

extern "C" int dahitra_pixel_decoder_train_bwd_ex(const void* dout, const float* xs, const float* tables, void* dx,
                                                  float* dtables_partial, int nimg, int npix, int heads, int depth, int pixel_major,
                                                  int act_dtype, void* stream) {
  const int eb = dh_act_bytes(act_dtype);
  DH_REQUIRE(eb > 0, DH_E_VARIANT);
  DH_REQUIRE(dout && xs && tables && dx && dtables_partial, DH_E_NULL);
  DH_REQUIRE(nimg > 0 && npix > 0 && depth > 0 && nimg <= 65535, DH_E_SHAPE);
  DH_REQUIRE(heads == 4 || heads == 8, DH_E_SHAPE);
  const int xal = pixel_major ? 16 : eb;
  DH_REQUIRE(dh_aligned16(tables) && dh_aligned(dout, xal) && dh_aligned(dx, xal), DH_E_ALIGN);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  return dh_act_dispatch(act_dtype, [&](auto t) {
    using TA = decltype(t);
    const TA* da = static_cast<const TA*>(dout);
    TA* xa = static_cast<TA*>(dx);
    if (pixel_major)
      return heads == 4 ? launch_bwd<16, true>(da, xs, tables, xa, dtables_partial, nimg, npix, depth, s)
                        : launch_bwd<32, true>(da, xs, tables, xa, dtables_partial, nimg, npix, depth, s);
    return heads == 4 ? launch_bwd<16, false>(da, xs, tables, xa, dtables_partial, nimg, npix, depth, s)
                      : launch_bwd<32, false>(da, xs, tables, xa, dtables_partial, nimg, npix, depth, s);
  });
}

extern "C" int dahitra_pixel_decoder_train_fwd(const float* x, const float* tables, float* xs, float* out, int nimg, int npix,
                                               int heads, int depth, int pixel_major, void* stream) {
  return dahitra_pixel_decoder_train_fwd_ex(x, tables, xs, out, nimg, npix, heads, depth, pixel_major, DH_ACT_F32, stream);
}

extern "C" int dahitra_pixel_decoder_train_bwd(const float* dout, const float* xs, const float* tables, float* dx,
                                               float* dtables_partial, int nimg, int npix, int heads, int depth, int pixel_major,
                                               void* stream) {
  return dahitra_pixel_decoder_train_bwd_ex(dout, xs, tables, dx, dtables_partial, nimg, npix, heads, depth, pixel_major,
                                            DH_ACT_F32, stream);
}
