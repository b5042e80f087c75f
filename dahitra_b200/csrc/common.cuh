// dahitra_b200 — shared device/host helpers (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include "../../include/dahitra_b200.h"

#ifndef __CUDA_ARCH_LIST__
#endif

#define DH_CHECK_LAUNCH()                                   \
  do {                                                      \
    cudaError_t e__ = cudaGetLastError();                   \
    if (e__ != cudaSuccess) return (int)e__;                \
  } while (0)

#define DH_REQUIRE(cond, code) \
  do {                         \
    if (!(cond)) return (code);\
  } while (0)

static inline bool dh_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline int dh_cdiv(int a, int b) { return (a + b - 1) / b; }

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// exact-erf GELU (nn.GELU() default; reference models/help_funcs.py:57)
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

// ---- internal launchers shared between the per-kernel C ABI and dahitra_forward ----------------
struct ConvArgs {
  const float* in0; const float* in1; int C0, C1;
  int N, inH, inW, up;           // stored input size; `up`=2 => virtual nearest x2 upsample
  int KH, KW, stride, pad, Cout;
  const float* w;                // [KH*KW*Cin][Cout]  (CUDA-core kernel)
  const float* wt;               // [Cout][KH*KW*Cin]  (tcgen05 kernel), may be NULL
  const float* bias; const float* res; int relu;
  float* out;
  // tcgen05 kernel only: "pixel-shuffle" store.  The conv has Cout = 4*32 channels = 4 output-pixel phases of
  // a nearest-x2-upsampled 3x3 conv (see engine.py: upsample_phase_filter); block j of 32 channels goes to
  // output pixel (2*oy + j/2, 2*ox + j%2) of a [N][2*inH][2*inW][32] tensor.
  int ps = 0;
  // tcgen05 kernel only: one tile per CTA instead of a persistent grid, so that the hardware scheduler can interleave
  // this launch with others (used for the head convolution that runs under the transformer levels on a side stream)
  int flat = 0;
};
// conv_tc3.cu: convolution over split16 activations (two FP16 planes hi | lo, see the file header)
struct Conv3Args {
  const void* in0; const void* in1; int C0, C1;      // split16 inputs (virtual concat of in0 | in1 along channels)
  int N, inH, inW;
  long long in0_plane = 0, in1_plane = 0;            // elements between the hi and lo planes (0: N*inH*inW*C; larger when in0 / in1
                                                     // are the first / second half of the images of one tensor)
  long long res_plane = 0, out_plane = 0;            // same for a split16 residual / output (0: N*OH*OW*Cout)
  int K, stride, Cout;                               // K = 1 or 3 (pad K/2); stride 1 or 2
  const void* wt16;                                  // FP16 filter planes h_w | l_w, each [Cout][K*K*Cin] (K-major)
  long long wt_plane_bytes;                          // bytes between the two planes
  const float* bias; const void* res; int res_split; // residual: fp32 NHWC or split16 (same shape as the output)
  int relu;
  void* out; int out_split;                          // fp32 NHWC or split16
  int ps = 0;                                        // pixel-shuffle store of a 32 -> 4x32 upsample convolution (fp32 output, or h16)
  int tok = 0;                                       // tokenizer epilogue (1x1, Cout 32): ReLU + store + per-tile softmax partials
  const float* wtok = nullptr; float* partials = nullptr;
  int force_stream = 0;                              // 1: never keep the filter resident in shared memory (A/B tests)
  int cg = 0;                                        // 0 = auto, 1 = single CTAs, 2 = CTA pairs (tcgen05 cta_group::2)
  int h16 = 0;                                       // 1: in0 / in1 and a split16 res / out are ONE FP16 plane each (in*_plane,
                                                     // res_plane, out_plane unused), the filter contributes h_w alone; no CTA pairs
};
bool dh_conv_tc3_eligible(const Conv3Args& a);
int dh_launch_conv_tc3(const Conv3Args& a, cudaStream_t s);
int dh_conv_tc3_tok_chunks(int H, int W);            // partial-softmax chunks per image the tok epilogue writes
// split.cu: fp32 NHWC <-> split16 planes, 3x3/s2 max pool on split16
int dh_launch_split_pack(const float* in, size_t n, void* out, cudaStream_t s);
int dh_launch_split_unpack(const void* in, size_t n, float* out, cudaStream_t s);
int dh_launch_maxpool_split(const void* in, int N, int H, int W, int C, void* out, cudaStream_t s);
int dh_launch_maxpool_h16(const void* in, int N, int H, int W, int C, void* out, cudaStream_t s);      // one FP16 plane
// programmatic dependent launch: attribute for cudaLaunchKernelEx (returns the number of attributes written: 0 or 1)
int dh_pdl_attr(cudaLaunchAttribute* at);
void dh_set_pdl(int on);
// launch with the programmatic-dependent-launch attribute when dahitra_forward asked for it (DH_FLAG_PDL): the kernel may
// start while its predecessor in the stream drains and must call pdl_wait() before touching anything that launch wrote
template <typename... KArgs, typename... Args>
static inline int dh_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  cfg.attrs = at; cfg.numAttrs = dh_pdl_attr(at);
  const cudaError_t e = cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
  if (e != cudaSuccess) return (int)e;
  DH_CHECK_LAUNCH();
  return 0;
}
#ifdef __CUDACC__
__device__ __forceinline__ void dh_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void dh_pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif
int dh_launch_conv_ffma(const ConvArgs& a, cudaStream_t s);
bool dh_conv_tc_eligible(const ConvArgs& a);
int dh_launch_conv_tc(const ConvArgs& a, cudaStream_t s);
bool dh_conv_tc2_eligible(const ConvArgs& a);                     // stride-1 halo-reuse kernel (conv_tc2.cu)
int dh_launch_conv_tc2(const ConvArgs& a, int xm, int cg, cudaStream_t s);
int dh_launch_stem(const float* x, long long xbs, int N, int H, int W, const float* w, const float* b, float* out, cudaStream_t s);
int dh_launch_stem_tc(const float* x, long long xbs, int N, int H, int W, const float* wtc, const float* b, float* out, int x3,
                      cudaStream_t s, long long split_plane_pitch = 0, const float* x_second = nullptr);
int dh_launch_maxpool(const float* in, int N, int H, int W, int C, float* out, cudaStream_t s);
int dh_launch_classifier(const float* in, int N, int H, int W, int nc, const float* w, const float* b,
                         float* logits, unsigned char* amax, cudaStream_t s);
int dh_launch_classifier_tma(const float* in, int N, int H, int W, int nc, const float* w, const float* b,
                             float* logits, unsigned char* amax, cudaStream_t s);
int dh_launch_classifier_h16(const void* in, int N, int H, int W, int nc, const float* w, const float* b,    // one FP16 plane in
                             float* logits, unsigned char* amax, cudaStream_t s);
int dh_launch_squeeze_tokens(const float* feat, int N, int npix, int Cin, const float* wsq, const float* wtok,
                             float* xs, float* partials, cudaStream_t s);
int dh_launch_token_encoder(const float* partials, int B, int nchunk, const float* enc, int heads, int add_pos,
                            float* mem, cudaStream_t s);
int dh_launch_decoder_tables(const float* mem, int B, int first_call, int ncalls, const float* dec, int heads, int depth,
                             float* tables, cudaStream_t s);
int dh_launch_decoder_tables_tc(const float* mem, int B, int first_call, int ncalls, const float* dec, int heads, int depth,
                                float* tables, cudaStream_t s);
int dh_launch_pixel_decoder_tc(const float* x, const float* pos, const float* tables, const float* pack, int nimg, int h,
                               int w, int heads, int depth, const float* skip, int skip_up, int x3, float* out,
                               cudaStream_t s);
int dh_launch_pixel_decoder(const float* x, const float* pos, const float* tables, const float* dec,
                            int nimg, int h, int w, int heads, int depth, const float* skip, int skip_up, float* out,
                            cudaStream_t s);
