/*
 * dahitra_b200 — C ABI of the sm_100a kernel library behind the drop-in `newUNetTrans` module.
 *
 * The reference (nka77/DAHiTra) is pure Python/PyTorch and has no FFI of its own; the boundary this
 * library sits behind is the nn.Module contract
 *     net = define_G(args, gpu_ids)            reference models/networks.py:130-168
 *     logits = net(x1, x2)                     reference models/networks.py:1321-1357
 * Each entry point below names the reference code whose arithmetic it replaces.  A reference
 * maintainer binds it with ctypes (see INTEGRATION.md); no torch types cross this interface.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless stated; the caller owns all memory (inputs, outputs,
 *     prepared weights, workspace).  The library never allocates or frees device memory and never synchronises.
 *     dahitra_forward forks two internal side streams off the caller's stream (event record / wait only, created on
 *     first use per host thread and device) and joins them before it returns control of the stream; DH_FLAG_SERIAL
 *     keeps everything on the caller's stream.
 *   - launches are asynchronous on `stream` (a cudaStream_t passed as void*), CUDA-graph capturable.
 *   - return value: 0 ok; <0 argument/shape/alignment error detected on the host before any launch
 *     (DH_E_*); >0 a cudaError_t reported by cudaGetLastError() after a launch.
 *   - internal activation layout is NHWC fp32 ("pixels x channels"); public inputs/outputs of
 *     dahitra_forward keep the reference layout (NCHW fp32).
 */
#ifndef DAHITRA_B200_H
#define DAHITRA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DAHITRA_ABI_VERSION 2

/* error codes (negative) */
#define DH_E_NULL      (-1)   /* a required pointer is NULL */
#define DH_E_SHAPE     (-2)   /* unsupported shape (e.g. H or W not a multiple of 32, B < 1) */
#define DH_E_ALIGN     (-3)   /* pointer not 16-byte aligned */
#define DH_E_WORKSPACE (-4)   /* workspace smaller than dahitra_workspace_bytes() */
#define DH_E_VARIANT   (-5)   /* unknown variant / flags */
#define DH_E_WEIGHTS   (-6)   /* weight table has the wrong number of slots or a NULL slot */

/* network variants */
#define DH_VARIANT_LEVIR 0    /* models/networks.py:1142-1357: 3 decoder passes per level, pos-emb on all levels */
#define DH_VARIANT_XBD   1    /* xBD_code/zoo/model_transformer_encoding.py:242-449 */

/* flags for dahitra_forward */
#define DH_FLAG_NONE        0
#define DH_FLAG_CONV_TC     1   /* route eligible convolutions through the tcgen05/TMEM/TMA implicit-GEMM kernel */
#define DH_FLAG_TC_3XTF32   2   /* with CONV_TC: error-compensated 3xTF32 (fp32-grade accuracy) instead of 1xTF32 */
#define DH_FLAG_TC_STRIDE2  4   /* with CONV_TC: also route the stride-2 convolutions (TMA element strides) */
#define DH_FLAG_DEC_TC      8   /* pixel decoder on tcgen05 (TF32 operands), decoder_tc.cu */
#define DH_FLAG_STEM_TC     16  /* 7x7 stem on tcgen05 (on-chip im2col), stem_tc.cu */
#define DH_FLAG_DEC_TC_X3   32  /* with DEC_TC: error-compensated 3xTF32 in the decoder (fp32-grade accuracy) */
#define DH_FLAG_CONV_TC_V1  64  /* with CONV_TC: force the per-tap TMA kernel (conv_tc.cu) instead of the halo-reuse one */
#define DH_FLAG_CONV_TC_2CTA 128 /* with CONV_TC: CTA pairs (tcgen05 cta_group::2, clusters of 2): M = 256 per MMA, half the filter traffic per SM */
#define DH_FLAG_SERIAL      256 /* keep every launch on the caller's stream (no fork of levels 4 / 3 onto the library's side streams) */
#define DH_FLAG_TC_X3_BF16  512 /* with TC_3XTF32: the two correction products of every conv as BF16 MMAs (half their cost) */
#define DH_FLAG_TC_BF16     1024 /* with CONV_TC: single-pass BF16 operands in the convolutions (fp32 storage and accumulation); overrides TC_3XTF32 */
#define DH_FLAG_TC_MAIN_F16 2048 /* with TC_3XTF32: main product of every conv in FP16 (K = 16 MMAs), both corrections in BF16; without it: single-pass FP16 operands */
#define DH_FLAG_TC_FOLD     4096 /* with TC_3XTF32 | TC_MAIN_F16: fold the f16(a).r_w correction into the main MMA (2N-wide filter tile); with TC_X3_BF16 the stem runs the same folded FP16 form */
#define DH_FLAG_EARLY_HEAD  8192 /* issue conv_layer2_0.0 right after the stem on a lowest-priority side stream, one tile per CTA */
#define DH_FLAG_ACT_SPLIT   16384 /* with the folded FP16 mode (TC_3XTF32 | TC_MAIN_F16 | TC_FOLD | STEM_TC | DEC_TC): activations that feed a
                                   * convolution are STORED as the split16 pair the MMAs consume (hi = f16(a), lo = f16(2^11 (a - hi)); 4 bytes
                                   * per element like fp32) and every convolution runs conv_tc3.cu: no splitter pass, TMA lands the operands;
                                   * the tokenizer's 1x1 squeeze runs on the tensor cores with the softmax partials in its epilogue */
#define DH_FLAG_PDL         32768 /* programmatic dependent launch between consecutive launches of a stream (prologues overlap the previous
                                   * launch's tail; every kernel waits with griddepcontrol.wait before touching its inputs) */
#define DH_FLAG_ACT_H16     65536 /* with CONV_TC | TC_MAIN_F16 | TC_STRIDE2 | STEM_TC | DEC_TC (and none of ACT_SPLIT, TC_3XTF32, TC_BF16,
                                   * CONV_TC_V1; dahitra_forward returns DH_E_VARIANT otherwise): every tensor the forward writes to its
                                   * workspace is stored as ONE FP16 plane (round to nearest, saturating at +-65504; 2 bytes per element)
                                   * except the tokenizer partials, token memories and decoder tables; single-pass FP16 convolutions on
                                   * conv_tc3.cu's single-plane form, FP16 max pools and classifier input.  Inputs and logits stay fp32 */
/* the modes dahitra_b200.engine.MODES names (DESIGN.md "Precision modes") */
#define DH_FLAGS_TF32X3     (DH_FLAG_CONV_TC | DH_FLAG_TC_3XTF32 | DH_FLAG_TC_X3_BF16 | DH_FLAG_TC_MAIN_F16 | DH_FLAG_TC_FOLD | DH_FLAG_TC_STRIDE2 | \
                             DH_FLAG_STEM_TC | DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3 | DH_FLAG_ACT_SPLIT | DH_FLAG_PDL)   /* default: every product error-compensated, fp32-grade */
#define DH_FLAGS_TF32       (DH_FLAG_CONV_TC | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3)   /* single-pass TF32 convs */
#define DH_FLAGS_F16        (DH_FLAGS_TF32 | DH_FLAG_TC_MAIN_F16)                    /* single-pass FP16 conv operands */
#define DH_FLAGS_BF16       (DH_FLAGS_TF32 | DH_FLAG_TC_BF16)                        /* single-pass BF16 conv operands */
#define DH_FLAGS_H16        (DH_FLAGS_F16 | DH_FLAG_ACT_H16 | DH_FLAG_PDL)           /* FP16 operands AND FP16 activation storage */

/* ---- prepared-weight table -------------------------------------------------------------------
 * dahitra_forward takes `const void* const* weights` with DH_W_COUNT slots, each a device pointer to
 * fp32 data prepared on the host side by dahitra_b200/engine.py (BN folded into conv weight/bias,
 * conv weights re-laid-out to [KH*KW*Cin][Cout], transformer products collapsed).  Slot meaning:
 */
enum dh_weight_slot {
  DH_W_STEM_W = 0, DH_W_STEM_B,                    /* resnet.conv1+bn1: [7*7*3][64] (r,s,ci major->minor), [64] */
  /* trunk 3x3 / 1x1 convs with their BN folded: weight [K][Cout], bias [Cout] */
  DH_W_L1_0_C1_W, DH_W_L1_0_C1_B, DH_W_L1_0_C2_W, DH_W_L1_0_C2_B,
  DH_W_L1_1_C1_W, DH_W_L1_1_C1_B, DH_W_L1_1_C2_W, DH_W_L1_1_C2_B,
  DH_W_L2_0_C1_W, DH_W_L2_0_C1_B, DH_W_L2_0_C2_W, DH_W_L2_0_C2_B, DH_W_L2_0_DS_W, DH_W_L2_0_DS_B,
  DH_W_L2_1_C1_W, DH_W_L2_1_C1_B, DH_W_L2_1_C2_W, DH_W_L2_1_C2_B,
  DH_W_L3_0_C1_W, DH_W_L3_0_C1_B, DH_W_L3_0_C2_W, DH_W_L3_0_C2_B, DH_W_L3_0_DS_W, DH_W_L3_0_DS_B,
  DH_W_L3_1_C1_W, DH_W_L3_1_C1_B, DH_W_L3_1_C2_W, DH_W_L3_1_C2_B,
  /* per level (5, 4, 3): squeeze [Cin][32]; token conv [32][4]; encoder pack; decoder pack;
   * decoder positional embedding [h*w][32] (NULL when the variant adds none); conv_decode [9*64][32] */
  DH_W_LV5_SQ, DH_W_LV5_TOK, DH_W_LV5_ENC, DH_W_LV5_DEC, DH_W_LV5_POS, DH_W_LV5_DECODE,
  DH_W_LV4_SQ, DH_W_LV4_TOK, DH_W_LV4_ENC, DH_W_LV4_DEC, DH_W_LV4_POS, DH_W_LV4_DECODE,
  DH_W_LV3_SQ, DH_W_LV3_TOK, DH_W_LV3_ENC, DH_W_LV3_DEC, DH_W_LV3_POS, DH_W_LV3_DECODE,
  /* UNet head */
  DH_W_CL4_W, DH_W_CL4_B, DH_W_CL3_W, DH_W_CL3_B, DH_W_CL2_W, DH_W_CL2_B,   /* conv_layer4/3/2: [9*32][32],[32] */
  DH_W_CL20A_W, DH_W_CL20A_B,                      /* conv_layer2_0.0 + BN: [9*128][128],[128] */
  DH_W_CL20B_W, DH_W_CL20B_B,                      /* conv_layer2_0.3: [9*128][32],[32] */
  DH_W_CLS_W, DH_W_CLS_B,                          /* classifier: [9][output_nc][32], [output_nc] */
  /* K-major copies of the filters the tcgen05 kernels take as their B operand (Cin a multiple of 32); same values
   * as the matching _W / _DECODE slot.  Layout: float [5][Cout][KH*KW*Cin] = TF32-rounded w | TF32-rounded remainder |
   * raw bits of a bf16 [2][Cout][K] array {bf16(w), bf16(w - plane 0)} (DH_FLAG_TC_X3_BF16) | raw bits of
   * {f16(w) saturated, bf16(w - f16(w))} (DH_FLAG_TC_MAIN_F16) | raw bits of {f16(2^11 (w - f16(w))), zeros}
   * (DH_FLAG_TC_FOLD): float [5][Cout][K] in total */
  DH_W_L1_0_C1_WT, DH_W_L1_0_C2_WT, DH_W_L1_1_C1_WT, DH_W_L1_1_C2_WT,
  DH_W_L2_0_C2_WT, DH_W_L2_1_C1_WT, DH_W_L2_1_C2_WT,
  DH_W_L3_0_C1_WT, DH_W_L3_0_C2_WT, DH_W_L3_0_DS_WT, DH_W_L3_1_C1_WT, DH_W_L3_1_C2_WT,
  DH_W_LV5_DECODE_WT, DH_W_LV4_DECODE_WT, DH_W_LV3_DECODE_WT,
  DH_W_CL20A_WT, DH_W_CL20B_WT,
  DH_W_L2_0_C1_WT, DH_W_L2_0_DS_WT,               /* the two stride-2 convs (TMA element strides) */
  /* conv_layer4/3/2 act on a nearest-x2-upsampled map.  On the tensor-core path each becomes ONE 3x3 conv
   * 32 -> 4*32 on the LOW-resolution map whose 4 channel blocks are the 4 output-pixel phases (filter taps
   * that coincide on the low-res grid are summed on the host): _PSWT [128][9*32] K-major, _PSB [128] */
  DH_W_CL4_PSWT, DH_W_CL4_PSB, DH_W_CL3_PSWT, DH_W_CL3_PSB, DH_W_CL2_PSWT, DH_W_CL2_PSB,
  /* tensor-core pixel decoder: per layer [W1f swz 32x32][W2 swz 32x32][b1f 32][cbA 32][cbM 32]
   * (DH_DECTC_LAYER_FLOATS), "swz" = K-major SWIZZLE_128B image of B[n][k] (W1f: n=hidden, k=channel, LN2
   * gamma folded; W2: n=channel, k=hidden); cbA/cbM = cumulative biases after the attention / MLP of the layer */
  DH_W_LV5_DECTC, DH_W_LV4_DECTC, DH_W_LV3_DECTC,
  DH_W_STEM_WTC,   /* stem filter for the tcgen05 stem; K ordered (ci, r, s8): 21 groups of 1 zero + 7 taps, padded to 192.  [0, 24576) floats: TF32 [hi, lo] x 6 K-step tiles of B[n=co 64][k 32] swz; [24576, 36864): bits of 3 K-step tiles of [f16(w) 64 rows ; f16(2^11 (w - f16 w)) 64 rows][k 64] swz; [36864, 43008): bits of 3 tiles of bf16(w)[64][k 64] swz */
  /* K-major split filters of the three 1x1 squeeze convolutions (same five planes as the other *_WT slots, [32][Cin]):
   * with DH_FLAG_ACT_SPLIT the squeeze + tokenizer partials run as a conv_tc3 launch */
  DH_W_LV5_SQ_WT, DH_W_LV4_SQ_WT, DH_W_LV3_SQ_WT,
  DH_W_COUNT
};

/* Encoder pack (floats), per level, heads = He:
 *   pos[8*32]  ln1_g[32] ln1_b[32]  Mqk[He][32 c][32 c']  MvoT[He][32 c'][32 c]  b_out[32]
 *   ln2_g[32] ln2_b[32]  W1t[32 c][32 o]  b1[32]  W2t[32 o][32 c]  b2[32]
 * Decoder pack (floats), per level, heads = Hd, per layer (stride DH_DEC_LAYER_FLOATS(Hd)):
 *   ln1_g[32] ln1_b[32]  MqkT[Hd][32 c'][32 c]  MovT[Hd][32 c'][32 c]  b_out[32]
 *   W1f[32 c][32 o] (ln2 gamma folded; ln2 beta folded into b1f)  b1f[32]  W2t[32 o][32 c]  b2[32]
 * with Mqk[h][c][c'] = dim^-0.5 * sum_d Wq[h*64+d][c] * Wk[h*64+d][c']   (c: query side, c': token side),
 *      Mvo[h][c][c'] = Mov[h][c][c'] = sum_d Wo[c][h*64+d] * Wv[h*64+d][c'];  "T" = stored transposed.
 */
#define DH_ENC_FLOATS(H)       (8*32 + 64 + 2*(H)*1024 + 32 + 64 + 1024 + 32 + 1024 + 32)
#define DH_DEC_LAYER_FLOATS(H) (64 + 2*(H)*1024 + 32 + 1024 + 32 + 1024 + 32)

int         dahitra_version(void);
const char* dahitra_error_string(int code);
const char* dahitra_weight_slot_name(int slot);          /* "DH_W_STEM_W", ... ; NULL if out of range */

/* ---- host-side weight preparation (no CUDA calls) ------------------------------------------------------------------
 * Reference-layout state_dict tensors -> the prepared slot table above: BatchNorm folding, filter re-layout and operand
 * planes, decoder collapse, swizzled images (csrc/prepare.cu; the same algebra as dahitra_b200/engine.py, in fp64).
 *   tensors        the checkpoint's tensors by their reference key (models/networks.py state_dict; xBD variant:
 *                  xBD_code/zoo/model_transformer_encoding.py), HOST pointers, contiguous, fp32 or fp64; unused keys ignored
 *   out            host buffer for all slots (fp32), or NULL to query the size
 *   slot_offsets   [DH_W_COUNT] float offset of every slot inside `out` (-1: slot absent, e.g. no positional embedding)
 * Returns the number of floats needed / written (> 0), or a negative DH_E_* code (DH_E_WEIGHTS: a required key is missing
 * or has the wrong number of elements).  Upload `out` with one copy; weights[i] = device_base + 4 * slot_offsets[i]. */
#define DH_DTYPE_F32 0
#define DH_DTYPE_F64 1
typedef struct dh_tensor { const char* name; const void* data; int dtype; int ndim; long long shape[4]; } dh_tensor;
long long dahitra_prepare_weights(const dh_tensor* tensors, int n_tensors, int variant, int output_nc,
                                  float* out, long long out_floats, long long* slot_offsets);

/* Bytes of scratch dahitra_forward needs for B pairs of HxW images (H, W multiples of 32). */
size_t dahitra_workspace_bytes(int variant, int B, int H, int W, int output_nc, int flags);

/* Whole bitemporal forward: replaces BASE_Transformer_UNet.forward (reference
 * models/networks.py:1321-1357; xBD variant model_transformer_encoding.py:409-449).
 *   x1, x2        (B,3,H,W) fp32 NCHW planes of the pre / post image; `x_batch_stride` = elements between
 *                 consecutive images of the same tensor (3*H*W for separate tensors, 6*H*W when x1/x2 are
 *                 the two halves of one (B,6,H,W) xBD input)
 *   logits        (B,output_nc,H,W) fp32 NCHW
 *   argmax_u8     optional (B,H,W) uint8 class map (torch.argmax(logits,1) tie rule: lowest index), or NULL
 */
int dahitra_forward(const void* const* weights, int n_weights,
                    const float* x1, const float* x2, long long x_batch_stride,
                    float* logits, unsigned char* argmax_u8,
                    void* workspace, size_t workspace_bytes,
                    int variant, int B, int H, int W, int output_nc, int flags, void* stream);

/* Diagnostic twin of dahitra_forward (same arguments, same arithmetic): records a CUDA event after every
 * launch, SYNCHRONISES `stream`, and fills host arrays (capacity `cap`) with each launch's device time (ms),
 * algorithmic FLOPs (2*MACs as the reference writes the op), algorithmic bytes (one read of its stored
 * inputs and weights + one write of its output) and a static name.  Returns the number of launches (> 0),
 * or an error (< 0; CUDA errors are reported as -(cudaError_t) - 1000).  Used by bench.py for the roofline. */
int dahitra_forward_profiled(const void* const* weights, int n_weights,
                             const float* x1, const float* x2, long long x_batch_stride,
                             float* logits, unsigned char* argmax_u8,
                             void* workspace, size_t workspace_bytes,
                             int variant, int B, int H, int W, int output_nc, int flags, void* stream,
                             int cap, float* ms, double* flops, double* bytes, const char** names);

/* ---- per-kernel entry points (block-level parity tests; NHWC fp32 activations) ---------------- */

/* Generic convolution: replaces nn.Conv2d(+folded BN)(+residual)(+ReLU) call sites, reference
 * models/resnet.py:57-73, models/networks.py:1194-1197,1243-1249, models/help_funcs.py:7-15.
 *   in0/in1   NHWC sources forming a virtual channel concat [in0 (C0) | in1 (C1)], C1 may be 0 (in1 NULL)
 *   up        1, or 2 = the input is virtually nearest-upsampled x2 first (nn.Upsample, networks.py:1102)
 *   w         [KH*KW*(C0+C1)][Cout], bias [Cout] or NULL, res NHWC [N][OH][OW][Cout] or NULL
 *   wt        K-major copy of the filter, [Cout][KH*KW*(C0+C1)], or NULL.  With flags & DH_FLAG_CONV_TC and a
 *             non-NULL wt, stride-1 un-upsampled convolutions (KH=KW in {1,3}, pad=KH/2, Cout in
 *             {32,64,128,256}) run on the tcgen05/TMEM/TMA implicit-GEMM kernel (TF32 operands, fp32
 *             accumulate); everything else runs on the fp32 CUDA-core kernel.
 *   C0, C1 multiples of 32; Cout multiple of 32.
 */
int dahitra_conv2d(const float* in0, const float* in1, int C0, int C1, int N, int inH, int inW, int up,
                   int KH, int KW, int stride, int pad, int Cout,
                   const float* w, const float* wt, const float* bias, const float* res, int relu,
                   float* out, int flags, void* stream);

/* nn.Upsample(scale_factor=2) (nearest) followed by a 3x3 pad-1 conv 32->32 (+bias)(+ReLU) — conv_layer4/3/2,
 * reference models/networks.py:1335-1336,1343-1344,1350-1351 — as ONE tcgen05 conv on the low-resolution map:
 *   in NHWC [N][inH][inW][32] -> out NHWC [N][2*inH][2*inW][32]
 *   pswt [2][128][9*32] K-major phase filter (hi, lo), psb [128] (see DH_W_CL*_PSWT / _PSB);
 *   flags: DH_FLAG_TC_3XTF32 and/or DH_FLAG_CONV_TC_V1 (DH_FLAG_CONV_TC is implied). */
int dahitra_conv2d_up2_tc(const float* in, int N, int inH, int inW, const float* pswt, const float* psb,
                          int relu, float* out, int flags, void* stream);

/* Stem: 7x7 stride-2 pad-3 conv 3->64 + folded BN + ReLU, NCHW planes in, NHWC out
 * (reference models/networks.py:1120-1122, models/resnet.py:150-153). */
int dahitra_stem(const float* x, long long x_batch_stride, int N, int H, int W,
                 const float* w, const float* bias, float* out, void* stream);

/* Same stem on the tensor cores: x3 = 0 TF32 operands, 1 error-compensated 3xTF32, 2 folded FP16 (fp32-grade for |x| <= 65504; the default mode's stem), 3 single-pass FP16 (the f16 / bf16 modes' stem); wtc = DH_W_STEM_WTC image.
 * x3 | 256 (forms 2 and 3): out receives split16 planes instead of fp32.
 * x3 | 512 (form 3 only): out receives one FP16 plane [N][H/2][W/2][64] (the h16 mode). */
int dahitra_stem_tc(const float* x, long long x_batch_stride, int N, int H, int W,
                    const float* wtc, const float* bias, float* out, int x3, void* stream);

/* MaxPool2d(3, stride 2, pad 1) on NHWC (reference models/networks.py:1123,1128). */
int dahitra_maxpool3x3s2(const float* in, int N, int H, int W, int C, float* out, void* stream);

/* Squeeze (1x1 conv + ReLU) fused with the tokenizer's spatial-softmax partial sums
 * (reference models/networks.py:1177-1184, 1273-1280).
 *   feat NHWC [N][npix][Cin] -> xs NHWC [N][npix][32]; partials [N][nchunk][4][34] = {max, sum, t[32]} per token,
 *   nchunk = ceil(npix/256) (one CTA of 128 threads covers 256 pixels). */
int dahitra_squeeze_tokens(const float* feat, int N, int npix, int Cin, const float* w_sq, const float* w_tok,
                           float* xs, float* partials, void* stream);

/* Token stage for B pairs: finishes the spatial softmax, adds pos-emb (if pos != 0), runs the 1-layer token
 * encoder (reference models/networks.py:1282-1286, 434-512) and emits the decoder memories
 *   mem [B][3][4][32] = {token1', token2', |token2' - token1'|}.
 * partials are laid out for 2B images: image b = pre image of pair b, image B+b = post image. */
int dahitra_token_encoder(const float* partials, int B, int nchunk, const float* enc_pack, int heads, int add_pos,
                          float* mem, void* stream);

/* Per (pair, call, layer) attention tables of the collapsed pixel decoder (see DESIGN.md §decoder):
 *   tables [B*ncalls][depth][DH_TAB_FLOATS(heads)] from mem [B][3][4][32] (calls first_call..first_call+ncalls-1). */
#define DH_TAB_FLOATS(H) (32*4*(H) + 4*(H) + 4*(H)*32 + 32)
int dahitra_decoder_tables(const float* mem, int B, int first_call, int ncalls, const float* dec_pack, int heads, int depth,
                           float* tables, void* stream);

/* Pixel decoder: replaces _forward_transformer_decoder + TransformerDecoder
 * (reference models/networks.py:1288-1295, models/help_funcs.py:66-114,170-186).
 *   x NHWC [nimg][npix][32]; pos [npix][32] or NULL; tables [nimg][depth][DH_TAB_FLOATS];
 *   skip: optional NHWC tensor added to the result: skip_up=2 -> [nimg][h/2][w/2][32] nearest-upsampled x2
 *         (networks.py:1329,1333), skip_up=1 -> [nimg][h][w][32] (networks.py:1340);
 *   out NHWC [nimg][npix][32]. */
int dahitra_pixel_decoder(const float* x, const float* pos, const float* tables, const float* dec_pack,
                          int nimg, int h, int w, int heads, int depth, const float* skip, int skip_up, float* out,
                          void* stream);

/* Tensor-core variants of the two decoder kernels (tcgen05, TF32 operands, fp32 accumulate in TMEM).
 *   tables: [nimg][depth][DH_TABTC_FLOATS] = per (image-call, layer) [TA swz 32x32][TB swz 32x32][cA 32]
 *   pack:   DH_W_LVk_DECTC (depth x DH_DECTC_LAYER_FLOATS)
 *   x3 != 0: error-compensated 3xTF32 (operands split hi + lo, three MMAs per product): fp32-grade accuracy.
 *   Every B operand is stored as a TF32-rounded "hi" tile plus a "lo" remainder tile:
 *     table record  [TA_hi][TB_hi][cA 32][TA_lo][TB_lo],  pack layer  [W1_hi][W2_hi][b1f][cbA][cbM][W1_lo][W2_lo] */
#define DH_TABTC_FLOATS        (1024 + 1024 + 32 + 2048)
#define DH_DECTC_LAYER_FLOATS  (1024 + 1024 + 32 + 32 + 32 + 2048)
int dahitra_decoder_tables_tc(const float* mem, int B, int first_call, int ncalls, const float* dec_pack, int heads,
                              int depth, float* tables, void* stream);
/* x3 | 256: out receives split16 planes instead of fp32.
 * x3 | 512: x, skip and out are one FP16 plane each (the h16 mode); the arithmetic inside is the same, out = f16(result). */
int dahitra_pixel_decoder_tc(const float* x, const float* pos, const float* tables, const float* dectc_pack,
                             int nimg, int h, int w, int heads, int depth, const float* skip, int skip_up, int x3,
                             float* out, void* stream);

/* ---- split16 activation format (DH_FLAG_ACT_SPLIT; conv_tc3.cu) --------------------------------------------------
 * A split16 tensor of n elements is two FP16 planes, hi at the pointer and lo n elements (2n bytes) later:
 *   hi = f16(a) saturating, lo = f16(2^11 (a - hi)),  a ~= hi + 2^-11 lo   (the same 4 bytes per element as fp32). */
int dahitra_split_pack(const float* in, long long n, void* out_split, void* stream);      /* n % 8 == 0 */
int dahitra_split_unpack(const void* in_split, long long n, float* out, void* stream);
/* MaxPool2d(3, 2, 1) on a split16 NHWC tensor (compares reconstructed values; the winner's planes are reproduced exactly) */
int dahitra_maxpool3x3s2_split(const void* in_split, int N, int H, int W, int C, void* out_split, void* stream);
/* MaxPool2d(3, 2, 1) on one FP16 NHWC plane (the h16 mode; exact, C % 8 == 0) */
int dahitra_maxpool3x3s2_h16(const void* in_h16, int N, int H, int W, int C, void* out_h16, void* stream);
/* Convolution over split16 inputs with all three partial products on FP16 MMAs (file header of conv_tc3.cu):
 *   in0 / in1      split16 NHWC sources (virtual channel concat, C1 may be 0); in*_plane = elements between their hi and lo
 *                  planes (0 = N*inH*inW*C; larger when they are sub-ranges of the images of one tensor)
 *   K in {1,3}, pad K/2, stride in {1,2}, Cout in {32,64,128,256}, C0 % 32 == C1 % 32 == 0
 *   wt             the conv's *_WT slot (float [5][Cout][K*K*Cin]); planes 3 and 4 hold h_w and l_w
 *   res            NULL, fp32 NHWC (res_split = 0) or split16 (res_split = 1); out fp32 NHWC or split16 (out_split)
 *   mode           0 plain | 1 pixel-shuffle store of a 32 -> 4x32 upsample conv (fp32 out [N][2inH][2inW][32]) |
 *                  2 tokenizer epilogue: no bias, ReLU, out = xs, partials [N][nchunk][4][34] with
 *                    nchunk = ceil(inH/16) * ceil(inW/8), w_tok [32][4]  (see dahitra_squeeze_tokens)
 *                  scheduling bits, OR-ed in (results do not depend on them): 16 = single CTAs, 32 = CTA pairs
 *                  (tcgen05 cta_group::2; default: chosen per shape), 64 = stream the filter from L2 even where it
 *                  would fit in shared memory
 *                  storage bit, OR-ed in: 128 = the h16 mode's format: in0, in1, a split res (res_split = 1) and a split out
 *                  (out_split = 1, also with the pixel-shuffle store) are ONE FP16 plane each, in*_plane is ignored, and only
 *                  h_w (plane 3) of the filter is read: one FP16 MMA per (tap, chunk, K step).  With 128 a CTA-pair request
 *                  (bit 32, or DAHITRA_TC3_CG) returns DH_E_VARIANT */
int dahitra_conv2d_split(const void* in0, const void* in1, int C0, int C1, long long in0_plane, long long in1_plane,
                         int N, int inH, int inW, int K, int stride, int Cout, const float* wt, const float* bias,
                         const void* res, int res_split, int relu, void* out, int out_split, int mode,
                         const float* w_tok, float* partials, void* stream);

/* Classifier 3x3 conv 32->nc (+bias), NHWC in, NCHW logits out, optional uint8 argmax map
 * (reference models/networks.py:1249,1355; harness argmax models/evaluator.py:89-92). */
int dahitra_classifier(const float* in, int N, int H, int W, int nc, const float* w, const float* bias,
                       float* logits, unsigned char* argmax_u8, void* stream);
/* The same classifier on one FP16 NHWC plane [N][H][W][32] (the h16 mode): TMA halo boxes of FP16, converted to fp32 on the
 * shared-memory read; fp32 sums, fp32 NCHW logits, uint8 argmax with the lowest-index tie rule. */
int dahitra_classifier_h16(const void* in_h16, int N, int H, int W, int nc, const float* w, const float* bias,
                           float* logits, unsigned char* argmax_u8, void* stream);

/* ---- training step (SURVEY.md §8 f4): pixel decoder forward that keeps the layer inputs + its hand-written backward ----------
 * Replaces, on the training route, the per-pixel arithmetic of reference models/help_funcs.py:66-114,170-186 and the
 * autograd graph eager PyTorch builds for it (models/trainer.py:247-262).  fp32 FMAs throughout.
 *   x, out, dout, dx  pixel_major = 0: channel-planar [nimg][32][npix] (the reference's NCHW tensors);
 *                     pixel_major = 1: [nimg][npix][32] (the same tensors in torch.channels_last memory format)
 *   tables            [nimg][depth][DH_TRAIN_TAB_FLOATS(heads)], per (image, layer), K = 4*heads, k = head*4 + token:
 *                       A [32][K] | c0 [K] | Bv [K][32] | bo [32] | W1 [32][32] | b1 [32] | W2 [32][32] | b2 [32]
 *                     (all matrices input-major; built by the host from Wq/Wk/Wv/Wo, the LayerNorm affines, the MLP and the
 *                     image's 4 memory tokens: dahitra_b200/modules.py PixelDecoder.train_tables)
 *   xs                [depth][nimg][32][npix]: the input of every layer, written by the forward and read by the backward
 *   dtables_partial   [nimg][dahitra_pixel_decoder_train_blocks(npix)][depth][DH_TRAIN_TAB_FLOATS]: every CTA WRITES the
 *                     table gradient of its pixels; the caller sums over the block axis (deterministic) */
#define DH_TRAIN_TAB_FLOATS(H) (65*4*(H) + 96 + 2048)
int dahitra_pixel_decoder_train_blocks(int npix);
int dahitra_pixel_decoder_train_fwd(const float* x, const float* tables, float* xs, float* out, int nimg, int npix,
                                    int heads, int depth, int pixel_major, void* stream);
int dahitra_pixel_decoder_train_bwd(const float* dout, const float* xs, const float* tables, float* dx,
                                    float* dtables_partial, int nimg, int npix, int heads, int depth, int pixel_major,
                                    void* stream);

/* Storage type of the per-pixel activations of the training kernels' _ex entry points (mixed-precision training: what autocast
 * hands over).  Values are converted to fp32 on load and all arithmetic stays fp32; 16-bit stores round to nearest even.  It
 * applies to x / out / dout / dx only: tables, xs, tokens, stats, w_tok and every partial stay fp32.  Alignment: pixel_major
 * tensors 16 bytes, planar ones one element.  An unknown act_dtype returns DH_E_VARIANT. */
#define DH_ACT_F32  0
#define DH_ACT_F16  1
#define DH_ACT_BF16 2
int dahitra_pixel_decoder_train_fwd_ex(const void* x, const float* tables, float* xs, void* out, int nimg, int npix,
                                       int heads, int depth, int pixel_major, int act_dtype, void* stream);
int dahitra_pixel_decoder_train_bwd_ex(const void* dout, const float* xs, const float* tables, void* dx,
                                       float* dtables_partial, int nimg, int npix, int heads, int depth, int pixel_major,
                                       int act_dtype, void* stream);

/* Semantic tokenizer of the training step: replaces reference models/networks.py:1273-1280 (_forward_semantic_tokens: 1x1 conv
 * 32 -> 4, softmax over the N pixels, einsum to 4 tokens) and its autograd graph.
 *   x, dx        [nimg][32][npix] (pixel_major = 0) or [nimg][npix][32] (pixel_major = 1): the post-ReLU squeeze output
 *   w_tok        [4][32] (conv_token_k.weight);  tokens / dtokens [nimg][4][32];  stats [nimg][4][2] = softmax max and sum
 *   partials     scratch [nimg][dahitra_tokenizer_train_chunks(npix)][4][34]
 *   dw_partial   [nimg][chunks][4][32]: WRITTEN per CTA; the caller sums over the first two axes (deterministic) */
int dahitra_tokenizer_train_chunks(int npix);
int dahitra_tokenizer_train_fwd(const float* x, const float* w_tok, float* partials, float* tokens, float* stats,
                                int nimg, int npix, int pixel_major, void* stream);
int dahitra_tokenizer_train_bwd(const float* x, const float* w_tok, const float* tokens, const float* stats,
                                const float* dtokens, float* dx, float* dw_partial, int nimg, int npix, int pixel_major,
                                void* stream);
/* the same with x / dx stored as act_dtype (DH_ACT_*) */
int dahitra_tokenizer_train_fwd_ex(const void* x, const float* w_tok, float* partials, float* tokens, float* stats,
                                   int nimg, int npix, int pixel_major, int act_dtype, void* stream);
int dahitra_tokenizer_train_bwd_ex(const void* x, const float* w_tok, const float* tokens, const float* stats,
                                   const float* dtokens, void* dx, float* dw_partial, int nimg, int npix, int pixel_major,
                                   int act_dtype, void* stream);

/* ---- next to the hot path (SURVEY.md §8 f1) ------------------------------------------------------------ */

/* Device-side confusion matrix: cm[g][p] += #{ i : gt[i] = g < nc, pred[i] = p } — replaces the per-batch
 * argmax -> .cpu().numpy() -> np.bincount of reference models/evaluator.py:95-104 / misc/metric_tool.py:141-158.
 *   pred, gt: uint8 class maps of n pixels (gt >= nc, e.g. 255, is ignored like the reference's mask);
 *   cm: device int64 [nc][nc], ACCUMULATED (zero it before the first call). */
int dahitra_confusion_matrix(const unsigned char* pred, const unsigned char* gt, long long n, int nc,
                             long long* cm, void* stream);

/* Input path (SURVEY.md 8 f2): uint8 HWC images [N][H][W][3] -> normalised fp32 NCHW on the device, bit-identical to the
 * reference loaders: kind 0 = (x/255 - 0.5)/0.5 (datasets/data_utils.py:104-111), kind 1 = x/127 - 1
 * (xBD_code/utils.py:112-116).  tile > 0 cuts every image into (H/tile)*(W/tile) square tiles in the reference's
 * patch order (data_utils.py:65-66, patch 0 at the origin) -> out [N*T][3][tile][tile]; tile = 0 keeps whole images. */
int dahitra_prepare_input_u8(const unsigned char* hwc, int N, int H, int W, int kind, int tile, float* nchw, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DAHITRA_B200_H */
