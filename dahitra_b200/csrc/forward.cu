// dahitra_b200 — C ABI + whole-network orchestration (launch sequence of the bitemporal forward).
#include "common.cuh"
#include <string.h>

// ----------------------------------------------------------------------------------------------------
// workspace plan
// ----------------------------------------------------------------------------------------------------
namespace {

struct Level {           // per transformer level (5, 4, 3)
  int cin, heads, depth, h, w;
  size_t xs, xd, dx, out, part, mem, tab;    // float offsets into the workspace
  int nchunk, nchunk3;
};

struct Plan {
  int B, H, W, nc, variant;
  size_t f2, p2, t4a, t4b, f4, t8a, t8b, t8c, f8, p8, t16a, t16b, t16c, f16;
  Level lv[3];
  size_t c4, c3, y20, o2, c2;
  size_t total_floats;
};

struct Bump {
  size_t off = 0;
  size_t take(size_t nfloats) {
    const size_t o = off;
    off += (nfloats + 63) & ~(size_t)63;   // 256-byte granules
    return o;
  }
};

bool make_plan(Plan& p, int variant, int B, int H, int W, int nc, int flags) {
  if (B < 1 || H < 32 || W < 32 || (H % 32) || (W % 32) || nc < 1 || nc > 8) return false;
  if (variant != DH_VARIANT_LEVIR && variant != DH_VARIANT_XBD) return false;
  p.B = B; p.H = H; p.W = W; p.nc = nc; p.variant = variant;
  const size_t N2 = 2 * (size_t)B;
  const size_t s2 = (size_t)(H / 2) * (W / 2), s4 = s2 / 4, s8 = s4 / 4, s16 = s8 / 4;
  Bump b;
  p.f2 = b.take(N2 * s2 * 64);
  p.p2 = b.take(N2 * s4 * 64);
  p.t4a = b.take(N2 * s4 * 64); p.t4b = b.take(N2 * s4 * 64); p.f4 = b.take(N2 * s4 * 64);
  p.t8a = b.take(N2 * s8 * 128); p.t8b = b.take(N2 * s8 * 128); p.t8c = b.take(N2 * s8 * 128); p.f8 = b.take(N2 * s8 * 128);
  p.p8 = b.take(N2 * s16 * 128);
  p.t16a = b.take(N2 * s16 * 256); p.t16b = b.take(N2 * s16 * 256); p.t16c = b.take(N2 * s16 * 256); p.f16 = b.take(N2 * s16 * 256);
  const int cins[3] = {256, 128, 64}, heads[3] = {4, 4, 8}, depths[3] = {4, 4, 8}, div[3] = {16, 8, 4};
  for (int i = 0; i < 3; ++i) {
    Level& L = p.lv[i];
    L.cin = cins[i]; L.heads = heads[i]; L.depth = depths[i]; L.h = H / div[i]; L.w = W / div[i];
    const size_t n = (size_t)L.h * L.w;
    L.nchunk = (int)((n + 255) / 256);                           // squeeze_tokens_kernel: one partial per 256 pixels
    L.nchunk3 = dh_conv_tc3_tok_chunks(L.h, L.w);                // conv_tc3 tok epilogue: one per 16 x 8 tile
    L.xs = b.take(N2 * n * 32);
    L.xd = b.take(N2 * n * 32);
    L.dx = b.take((size_t)B * n * 32);
    L.out = b.take((size_t)B * n * 32);
    L.part = b.take(N2 * (size_t)(L.nchunk3 > L.nchunk ? L.nchunk3 : L.nchunk) * 4 * 34);
    L.mem = b.take((size_t)B * 3 * 128);
    L.tab = b.take((size_t)3 * B * L.depth * (DH_TAB_FLOATS(L.heads) > DH_TABTC_FLOATS ? DH_TAB_FLOATS(L.heads) : DH_TABTC_FLOATS));
  }
  p.c4 = b.take((size_t)B * s4 * 32);
  // The head's tensors reuse trunk buffers that are dead by then (every launch that reads them has been joined into the main
  // stream before the head starts; a programmatic dependent launch only overlaps a kernel with its direct predecessor):
  //   C3  (conv_layer3 out)      <- T8a | T8b          Y20 (conv_layer2_0.0 out) <- P2 | T4a | T4b | F4
  //   O2  (conv_layer2_0.3 out)  <- T8c | F8           C2  (conv_layer2 out)     <- F2 (last read by conv_layer2_0.0)
  // 13 -> 8 units of B * (H/2) * (W/2) * 64 floats: 3.5 -> 2.1 GB at 64 LEVIR pairs.  DH_FLAG_EARLY_HEAD issues conv_layer2_0.0
  // right after the stem, so Y20 keeps its own buffer under that flag.
  const size_t n_c3 = (size_t)B * s2 * 32, n_y20 = (size_t)B * s2 * 128, n_c2 = (size_t)B * H * W * 32;
  const bool early_head = (flags & DH_FLAG_EARLY_HEAD) != 0;
  p.c3 = (p.t8c - p.t8a >= n_c3) ? p.t8a : b.take(n_c3);
  p.o2 = (p.p8 - p.t8c >= n_c3) ? p.t8c : b.take(n_c3);
  p.y20 = (!early_head && p.t8a - p.p2 >= n_y20) ? p.p2 : b.take(n_y20);
  p.c2 = (p.p2 - p.f2 >= n_c2) ? p.f2 : b.take(n_c2);
  p.total_floats = b.off;
  return true;
}

const char* kSlotNames[DH_W_COUNT] = {
  "DH_W_STEM_W", "DH_W_STEM_B",
  "DH_W_L1_0_C1_W", "DH_W_L1_0_C1_B", "DH_W_L1_0_C2_W", "DH_W_L1_0_C2_B",
  "DH_W_L1_1_C1_W", "DH_W_L1_1_C1_B", "DH_W_L1_1_C2_W", "DH_W_L1_1_C2_B",
  "DH_W_L2_0_C1_W", "DH_W_L2_0_C1_B", "DH_W_L2_0_C2_W", "DH_W_L2_0_C2_B", "DH_W_L2_0_DS_W", "DH_W_L2_0_DS_B",
  "DH_W_L2_1_C1_W", "DH_W_L2_1_C1_B", "DH_W_L2_1_C2_W", "DH_W_L2_1_C2_B",
  "DH_W_L3_0_C1_W", "DH_W_L3_0_C1_B", "DH_W_L3_0_C2_W", "DH_W_L3_0_C2_B", "DH_W_L3_0_DS_W", "DH_W_L3_0_DS_B",
  "DH_W_L3_1_C1_W", "DH_W_L3_1_C1_B", "DH_W_L3_1_C2_W", "DH_W_L3_1_C2_B",
  "DH_W_LV5_SQ", "DH_W_LV5_TOK", "DH_W_LV5_ENC", "DH_W_LV5_DEC", "DH_W_LV5_POS", "DH_W_LV5_DECODE",
  "DH_W_LV4_SQ", "DH_W_LV4_TOK", "DH_W_LV4_ENC", "DH_W_LV4_DEC", "DH_W_LV4_POS", "DH_W_LV4_DECODE",
  "DH_W_LV3_SQ", "DH_W_LV3_TOK", "DH_W_LV3_ENC", "DH_W_LV3_DEC", "DH_W_LV3_POS", "DH_W_LV3_DECODE",
  "DH_W_CL4_W", "DH_W_CL4_B", "DH_W_CL3_W", "DH_W_CL3_B", "DH_W_CL2_W", "DH_W_CL2_B",
  "DH_W_CL20A_W", "DH_W_CL20A_B", "DH_W_CL20B_W", "DH_W_CL20B_B", "DH_W_CLS_W", "DH_W_CLS_B",
  "DH_W_L1_0_C1_WT", "DH_W_L1_0_C2_WT", "DH_W_L1_1_C1_WT", "DH_W_L1_1_C2_WT",
  "DH_W_L2_0_C2_WT", "DH_W_L2_1_C1_WT", "DH_W_L2_1_C2_WT",
  "DH_W_L3_0_C1_WT", "DH_W_L3_0_C2_WT", "DH_W_L3_0_DS_WT", "DH_W_L3_1_C1_WT", "DH_W_L3_1_C2_WT",
  "DH_W_LV5_DECODE_WT", "DH_W_LV4_DECODE_WT", "DH_W_LV3_DECODE_WT", "DH_W_CL20A_WT", "DH_W_CL20B_WT",
  "DH_W_L2_0_C1_WT", "DH_W_L2_0_DS_WT",
  "DH_W_CL4_PSWT", "DH_W_CL4_PSB", "DH_W_CL3_PSWT", "DH_W_CL3_PSB", "DH_W_CL2_PSWT", "DH_W_CL2_PSB",
  "DH_W_LV5_DECTC", "DH_W_LV4_DECTC", "DH_W_LV3_DECTC", "DH_W_STEM_WTC",
  "DH_W_LV5_SQ_WT", "DH_W_LV4_SQ_WT", "DH_W_LV3_SQ_WT"};

// filter slot -> slot of its K-major copy (or -1)
int wt_slot_of(int wslot) {
  switch (wslot) {
    case DH_W_L1_0_C1_W: return DH_W_L1_0_C1_WT; case DH_W_L1_0_C2_W: return DH_W_L1_0_C2_WT;
    case DH_W_L1_1_C1_W: return DH_W_L1_1_C1_WT; case DH_W_L1_1_C2_W: return DH_W_L1_1_C2_WT;
    case DH_W_L2_0_C2_W: return DH_W_L2_0_C2_WT; case DH_W_L2_1_C1_W: return DH_W_L2_1_C1_WT;
    case DH_W_L2_1_C2_W: return DH_W_L2_1_C2_WT;
    case DH_W_L3_0_C1_W: return DH_W_L3_0_C1_WT; case DH_W_L3_0_C2_W: return DH_W_L3_0_C2_WT;
    case DH_W_L3_0_DS_W: return DH_W_L3_0_DS_WT; case DH_W_L3_1_C1_W: return DH_W_L3_1_C1_WT;
    case DH_W_L3_1_C2_W: return DH_W_L3_1_C2_WT;
    case DH_W_LV5_DECODE: return DH_W_LV5_DECODE_WT; case DH_W_LV4_DECODE: return DH_W_LV4_DECODE_WT;
    case DH_W_LV3_DECODE: return DH_W_LV3_DECODE_WT;
    case DH_W_CL20A_W: return DH_W_CL20A_WT; case DH_W_CL20B_W: return DH_W_CL20B_WT;
    case DH_W_L2_0_C1_W: return DH_W_L2_0_C1_WT; case DH_W_L2_0_DS_W: return DH_W_L2_0_DS_WT;
    default: return -1;
  }
}

}  // namespace

// ----------------------------------------------------------------------------------------------------
// C ABI — utilities
// ----------------------------------------------------------------------------------------------------
extern "C" int dahitra_version(void) { return DAHITRA_ABI_VERSION; }

extern "C" const char* dahitra_error_string(int code) {
  switch (code) {
    case 0: return "ok";
    case DH_E_NULL: return "dahitra: required pointer is NULL";
    case DH_E_SHAPE: return "dahitra: unsupported shape";
    case DH_E_ALIGN: return "dahitra: pointer not 16-byte aligned";
    case DH_E_WORKSPACE: return "dahitra: workspace too small";
    case DH_E_VARIANT: return "dahitra: unknown variant or flags";
    case DH_E_WEIGHTS: return "dahitra: malformed weight table";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "dahitra: unknown error";
  }
}

extern "C" const char* dahitra_weight_slot_name(int slot) {
  return (slot >= 0 && slot < DH_W_COUNT) ? kSlotNames[slot] : nullptr;
}

extern "C" size_t dahitra_workspace_bytes(int variant, int B, int H, int W, int output_nc, int flags) {
  Plan p;
  if (!make_plan(p, variant, B, H, W, output_nc, flags)) return 0;
  return p.total_floats * sizeof(float);
}

// ----------------------------------------------------------------------------------------------------
// C ABI — per-kernel entry points
// ----------------------------------------------------------------------------------------------------
static int conv_dispatch(const ConvArgs& a, int flags, cudaStream_t s) {
  if (flags & DH_FLAG_CONV_TC) {
    // halo-reuse kernel (1xTF32 or error-compensated 3xTF32; stride 2 through the four phase images), or the older
    // per-tap TMA kernel (1xTF32) when DH_FLAG_CONV_TC_V1 asks for it.  Stride-2 convs need DH_FLAG_TC_STRIDE2.
    const bool stride_ok = a.stride == 1 || (flags & DH_FLAG_TC_STRIDE2);
    if (stride_ok && !(flags & DH_FLAG_CONV_TC_V1) && dh_conv_tc2_eligible(a))
      return dh_launch_conv_tc2(a, (flags & DH_FLAG_TC_BF16) ? 3 : (flags & DH_FLAG_TC_3XTF32) ? ((flags & DH_FLAG_TC_MAIN_F16) ? ((flags & DH_FLAG_TC_FOLD) ? 6 : 4) : (flags & DH_FLAG_TC_X3_BF16) ? 2 : 1)
                                                            : ((flags & DH_FLAG_TC_MAIN_F16) ? 5 : 0),
                                (flags & DH_FLAG_CONV_TC_2CTA) ? 2 : 1, s);
    if (stride_ok && dh_conv_tc_eligible(a)) return dh_launch_conv_tc(a, s);
  }
  return dh_launch_conv_ffma(a, s);
}

extern "C" int dahitra_conv2d(const float* in0, const float* in1, int C0, int C1, int N, int inH, int inW, int up,
                              int KH, int KW, int stride, int pad, int Cout, const float* w, const float* wt,
                              const float* bias, const float* res, int relu, float* out, int flags, void* stream) {
  ConvArgs a{in0, in1, C0, C1, N, inH, inW, up, KH, KW, stride, pad, Cout, w, wt, bias, res, relu, out};
  return conv_dispatch(a, flags, (cudaStream_t)stream);
}
extern "C" int dahitra_conv2d_up2_tc(const float* in, int N, int inH, int inW, const float* pswt, const float* psb,
                                     int relu, float* out, int flags, void* stream) {
  ConvArgs a{in, nullptr, 32, 0, N, inH, inW, 1, 3, 3, 1, 1, 128, nullptr, pswt, psb, nullptr, relu, out};
  a.ps = 1;
  DH_REQUIRE(dh_conv_tc_eligible(a), DH_E_SHAPE);
  return conv_dispatch(a, flags | DH_FLAG_CONV_TC, (cudaStream_t)stream);
}
extern "C" int dahitra_stem(const float* x, long long xbs, int N, int H, int W, const float* w, const float* bias,
                            float* out, void* stream) {
  return dh_launch_stem(x, xbs, N, H, W, w, bias, out, (cudaStream_t)stream);
}
extern "C" int dahitra_stem_tc(const float* x, long long xbs, int N, int H, int W, const float* wtc, const float* bias,
                               float* out, int x3, void* stream) {
  return dh_launch_stem_tc(x, xbs, N, H, W, wtc, bias, out, x3, (cudaStream_t)stream);
}
extern "C" int dahitra_maxpool3x3s2(const float* in, int N, int H, int W, int C, float* out, void* stream) {
  return dh_launch_maxpool(in, N, H, W, C, out, (cudaStream_t)stream);
}
extern "C" int dahitra_squeeze_tokens(const float* feat, int N, int npix, int Cin, const float* w_sq, const float* w_tok,
                                      float* xs, float* partials, void* stream) {
  return dh_launch_squeeze_tokens(feat, N, npix, Cin, w_sq, w_tok, xs, partials, (cudaStream_t)stream);
}
extern "C" int dahitra_token_encoder(const float* partials, int B, int nchunk, const float* enc_pack, int heads,
                                     int add_pos, float* mem, void* stream) {
  return dh_launch_token_encoder(partials, B, nchunk, enc_pack, heads, add_pos, mem, (cudaStream_t)stream);
}
extern "C" int dahitra_decoder_tables(const float* mem, int B, int first_call, int ncalls, const float* dec_pack,
                                      int heads, int depth, float* tables, void* stream) {
  return dh_launch_decoder_tables(mem, B, first_call, ncalls, dec_pack, heads, depth, tables, (cudaStream_t)stream);
}
extern "C" int dahitra_pixel_decoder(const float* x, const float* pos, const float* tables, const float* dec_pack,
                                     int nimg, int h, int w, int heads, int depth, const float* skip, int skip_up,
                                     float* out, void* stream) {
  return dh_launch_pixel_decoder(x, pos, tables, dec_pack, nimg, h, w, heads, depth, skip, skip_up, out,
                                 (cudaStream_t)stream);
}
extern "C" int dahitra_decoder_tables_tc(const float* mem, int B, int first_call, int ncalls, const float* dec_pack,
                                         int heads, int depth, float* tables, void* stream) {
  return dh_launch_decoder_tables_tc(mem, B, first_call, ncalls, dec_pack, heads, depth, tables, (cudaStream_t)stream);
}
extern "C" int dahitra_pixel_decoder_tc(const float* x, const float* pos, const float* tables, const float* dectc_pack,
                                        int nimg, int h, int w, int heads, int depth, const float* skip, int skip_up,
                                        int x3, float* out, void* stream) {
  return dh_launch_pixel_decoder_tc(x, pos, tables, dectc_pack, nimg, h, w, heads, depth, skip, skip_up, x3, out,
                                    (cudaStream_t)stream);
}
extern "C" int dahitra_split_pack(const float* in, long long n, void* out, void* stream) {
  return dh_launch_split_pack(in, (size_t)n, out, (cudaStream_t)stream);
}
extern "C" int dahitra_split_unpack(const void* in, long long n, float* out, void* stream) {
  return dh_launch_split_unpack(in, (size_t)n, out, (cudaStream_t)stream);
}
extern "C" int dahitra_maxpool3x3s2_split(const void* in, int N, int H, int W, int C, void* out, void* stream) {
  return dh_launch_maxpool_split(in, N, H, W, C, out, (cudaStream_t)stream);
}
extern "C" int dahitra_conv2d_split(const void* in0, const void* in1, int C0, int C1, long long in0_plane, long long in1_plane,
                                    int N, int inH, int inW, int K, int stride, int Cout, const float* wt, const float* bias,
                                    const void* res, int res_split, int relu, void* out, int out_split, int mode,
                                    const float* w_tok, float* partials, void* stream) {
  DH_REQUIRE(wt, DH_E_NULL);
  const int h16 = (mode & 128) ? 1 : 0;                              // storage format: one FP16 plane instead of split16
  const int sched = mode & ~(3 | 128);                               // scheduling bits (do not change results)
  mode &= 3;
  DH_REQUIRE(mode <= 2 && !(sched & ~(16 | 32 | 64)), DH_E_VARIANT);
  Conv3Args a{};
  a.h16 = h16;
  a.cg = (sched & 32) ? 2 : ((sched & 16) ? 1 : 0);
  a.force_stream = (sched & 64) ? 1 : 0;
  a.in0 = in0; a.in1 = in1; a.C0 = C0; a.C1 = C1; a.N = N; a.inH = inH; a.inW = inW; a.in0_plane = in0_plane; a.in1_plane = in1_plane;
  a.K = K; a.stride = stride; a.Cout = Cout;
  const size_t plane = (size_t)Cout * K * K * (C0 + C1);            // floats per plane of the *_WT slot
  a.wt16 = wt + 3 * plane; a.wt_plane_bytes = (long long)plane * 4;
  a.bias = bias; a.res = res; a.res_split = res_split; a.relu = relu; a.out = out; a.out_split = out_split;
  a.ps = mode == 1; a.tok = mode == 2; a.wtok = w_tok; a.partials = partials;
  return dh_launch_conv_tc3(a, (cudaStream_t)stream);
}
extern "C" int dahitra_classifier(const float* in, int N, int H, int W, int nc, const float* w, const float* bias,
                                  float* logits, unsigned char* argmax_u8, void* stream) {
  return dh_launch_classifier(in, N, H, W, nc, w, bias, logits, argmax_u8, (cudaStream_t)stream);
}
extern "C" int dahitra_maxpool3x3s2_h16(const void* in, int N, int H, int W, int C, void* out, void* stream) {
  return dh_launch_maxpool_h16(in, N, H, W, C, out, (cudaStream_t)stream);
}
extern "C" int dahitra_classifier_h16(const void* in, int N, int H, int W, int nc, const float* w, const float* bias,
                                      float* logits, unsigned char* argmax_u8, void* stream) {
  return dh_launch_classifier_h16(in, N, H, W, nc, w, bias, logits, argmax_u8, (cudaStream_t)stream);
}

// ----------------------------------------------------------------------------------------------------
// programmatic dependent launch switch (per host thread; set by dahitra_forward from DH_FLAG_PDL for its own launches)
// ----------------------------------------------------------------------------------------------------
namespace { thread_local int g_pdl = 0; }
void dh_set_pdl(int on) { g_pdl = on; }
int dh_pdl_attr(cudaLaunchAttribute* at) {
  if (!g_pdl) return 0;
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  return 1;
}

// ----------------------------------------------------------------------------------------------------
// per-launch profiler (diagnostic; used by bench.py for the roofline of the dominant kernel)
// ----------------------------------------------------------------------------------------------------
namespace {
constexpr int PROF_MAX = 160;
struct ProfRec { const char* name; double flops, bytes; };
struct Profiler {
  bool on = false, created = false;
  int n = 0;
  cudaEvent_t ev[PROF_MAX + 1];
  ProfRec rec[PROF_MAX];
};
thread_local Profiler g_prof;

inline void prof_mark(cudaStream_t s, const char* name, double flops, double bytes) {
  if (!g_prof.on || g_prof.n >= PROF_MAX) return;
  g_prof.rec[g_prof.n] = {name, flops, bytes};
  ++g_prof.n;
  cudaEventRecord(g_prof.ev[g_prof.n], s);
}
}  // namespace

// ----------------------------------------------------------------------------------------------------
// side streams: the token / decoder chains of levels 4 and 3 do not depend on level 5, and most of their kernels are
// too small to fill 148 SMs, so they are forked onto two auxiliary streams after the trunk and joined before the
// first launch that needs them (event record / wait only: asynchronous, graph-capturable, no host synchronisation).
// One set per (host thread, device), created on first use and kept for the life of the thread.
// ----------------------------------------------------------------------------------------------------
namespace {
struct AuxStreams {
  bool ok = false;
  cudaStream_t st[2], low;                 // low: lowest priority, for the head convolution that fills idle SMs
  cudaEvent_t fork, join[2], fork_low, join_low;
};
AuxStreams* aux_streams() {
  thread_local AuxStreams per_dev[16];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 16) return nullptr;
  AuxStreams& a = per_dev[dev];
  if (!a.ok) {
    bool good = cudaEventCreateWithFlags(&a.fork, cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; i < 2 && good; ++i)
      good = cudaStreamCreateWithFlags(&a.st[i], cudaStreamNonBlocking) == cudaSuccess &&
             cudaEventCreateWithFlags(&a.join[i], cudaEventDisableTiming) == cudaSuccess;
    if (good) {
      int lo = 0, hi = 0;
      cudaDeviceGetStreamPriorityRange(&lo, &hi);                 // lo = numerically largest = least priority
      good = cudaStreamCreateWithPriority(&a.low, cudaStreamNonBlocking, lo) == cudaSuccess &&
             cudaEventCreateWithFlags(&a.fork_low, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&a.join_low, cudaEventDisableTiming) == cudaSuccess;
    }
    if (!good) { cudaGetLastError(); return nullptr; }
    a.ok = true;
  }
  return &a;
}
}  // namespace

// ----------------------------------------------------------------------------------------------------
// whole forward
// ----------------------------------------------------------------------------------------------------
#define DH_STEP(name, fl, by, expr)        \
  do {                                     \
    const int rc__ = (expr);               \
    if (rc__ != 0) return rc__;            \
    prof_mark(s, name, (fl), (by));        \
  } while (0)

// ----------------------------------------------------------------------------------------------------
// Whole forward on split16 activations (DH_FLAG_ACT_SPLIT, the default fp32-grade mode).  Same launch order and the same
// reference semantics as the fp32-storage path below; what differs is the storage format of every tensor a convolution
// reads (two FP16 planes hi | lo in the buffer an fp32 tensor of that shape would occupy — the workspace plan is shared)
// and the kernels: conv_tc3 for every convolution including the tokenizer's 1x1 squeeze, the split16 max pool, and the
// stem / pixel decoder writing split16 where a convolution consumes their output.
//   split16: F2, P2, T4*, F4, T8*, F8, P8, T16*, F16, Y20, O2, decoder outputs read by a conv (XD; OUT of levels 4, 3),
//            XS in the xBD variant (read by conv_decode)
//   fp32:    XS (LEVIR: read by the decoder), DX, OUT of level 5 (a decoder skip), C4, C3, C2, logits
// The same sequence runs the h16 mode (DH_FLAG_ACT_H16): EVERY tensor listed above is stored as one FP16 plane (hi alone, 2 bytes
// per element, in half the buffer), the convolutions take the single-plane form of conv_tc3 (one MMA per (tap, chunk, K step)),
// the max pools and the classifier read FP16; the tokenizer partials, token memories and decoder tables stay fp32.  The
// algorithmic byte counts of the profiler use 2 bytes per element for those tensors (and for the h_w filter plane).
// ----------------------------------------------------------------------------------------------------
namespace {
int forward_split(const Plan& p, const void* const* weights, const float* x1, const float* x2, long long x_batch_stride,
                  float* logits, unsigned char* argmax_u8, float* ws, int variant, int B, int H, int W, int output_nc, int flags,
                  cudaStream_t s_main) {
  cudaStream_t s = s_main;
  auto Wt = [&](int slot) { return (const float*)weights[slot]; };
  const int N2 = 2 * B;
  const int h2 = H / 2, w2 = W / 2, h4 = H / 4, w4 = W / 4, h8 = H / 8, w8 = W / 8, h16 = H / 16, w16 = W / 16;
  const bool one = (flags & DH_FLAG_ACT_H16) != 0;     // one FP16 plane per tensor (every res / out below is then FP16)
  const double eb = one ? 2.0 : 4.0;                   // stored bytes per element of the tensors listed above
  // conv over split16 inputs.  wts: the filter's *_WT (or _PSWT) slot; in_plane: elements between the hi / lo planes of in0 / in1
  auto conv3 = [&](const char* name, const float* in0, const float* in1, int C0, int C1, long long in_plane, int N, int inH, int inW,
                   int K, int stride, int Cout, int wts, int bslot, const float* res, int res_split, int relu, float* out,
                   int out_split, int ps) -> int {
    Conv3Args a{};
    a.in0 = in0; a.in1 = in1; a.C0 = C0; a.C1 = C1; a.N = N; a.inH = inH; a.inW = inW; a.in0_plane = in_plane; a.in1_plane = in_plane;
    a.K = K; a.stride = stride; a.Cout = Cout;
    const size_t plane = (size_t)Cout * K * K * (C0 + C1);
    a.wt16 = Wt(wts) + 3 * plane; a.wt_plane_bytes = (long long)plane * 4;
    a.bias = bslot >= 0 ? Wt(bslot) : nullptr; a.res = res; a.res_split = one ? 1 : res_split; a.relu = relu; a.out = out;
    a.out_split = one ? 1 : out_split;
    a.ps = ps; a.h16 = one;
    const int rc = dh_launch_conv_tc3(a, s);
    if (rc != 0) return rc;
    const double OH = (double)inH / stride, OW = (double)inW / stride, Cin = C0 + C1;
    const double cout_alg = ps ? 32.0 : Cout, up = ps ? 2.0 : 1.0;       // as written: a 3x3 conv 32 -> 32 on the upsampled map
    const double fl = 2.0 * N * OH * up * OW * up * cout_alg * K * K * Cin;
    const double by = eb * ((double)N * inH * inW * Cin + (double)N * OH * up * OW * up * cout_alg * (res ? 2 : 1) + (double)K * K * Cin * cout_alg);
    prof_mark(s, name, fl, by);
    return 0;
  };
#define DH_CONV3(...)                     \
  do {                                    \
    const int rc__ = conv3(__VA_ARGS__);  \
    if (rc__ != 0) return rc__;           \
  } while (0)

  // ---- Siamese trunk on 2B images: [pre batch | post batch]  (reference networks.py:1118-1138, 1323-1324)
  // F2 is ONE split16 tensor of 2B images; the stem runs once per image set and writes its half of both planes.
  auto H16 = [](float* p) { return reinterpret_cast<uint16_t*>(p); };
  float* F2 = ws + p.f2;
  const size_t f2_half = (size_t)B * h2 * w2 * 64;
  const long long f2_plane = (long long)N2 * h2 * w2 * 64;
  float* F2post = reinterpret_cast<float*>(H16(F2) + f2_half);             // hi plane of the post images
  const double stem_fl = 2.0 * B * h2 * w2 * 64 * 147;
  const double stem_by = one ? B * (4.0 * 3 * H * W + 2.0 * h2 * w2 * 64) : 4.0 * B * ((double)3 * H * W + (double)h2 * w2 * 64);
  const int stem_mode = one ? 3 | 512 : ((flags & DH_FLAG_TC_3XTF32) ? 2 : 3) | 256;
  // one launch over both image sets (pre images first): x2 is addressed through a second tensor map
  DH_STEP("stem", 2.0 * stem_fl, 2.0 * stem_by,
          dh_launch_stem_tc(x1, x_batch_stride, B, H, W, Wt(DH_W_STEM_WTC), Wt(DH_W_STEM_B), F2, stem_mode, s, f2_plane, x2));
  float* P2 = ws + p.p2;
  auto maxpool = [&](const float* in, int hh, int ww, int C, float* out) {
    return one ? dh_launch_maxpool_h16(in, N2, hh, ww, C, out, s) : dh_launch_maxpool_split(in, N2, hh, ww, C, out, s);
  };
  DH_STEP("maxpool_2", 0.0, eb * N2 * 64 * ((double)h2 * w2 + (double)h4 * w4), maxpool(F2, h2, w2, 64, P2));
  float *T4a = ws + p.t4a, *T4b = ws + p.t4b, *F4 = ws + p.f4;
  DH_CONV3("layer1.0.conv1", P2, nullptr, 64, 0, 0, N2, h4, w4, 3, 1, 64, DH_W_L1_0_C1_WT, DH_W_L1_0_C1_B, nullptr, 0, 1, T4a, 1, 0);
  DH_CONV3("layer1.0.conv2", T4a, nullptr, 64, 0, 0, N2, h4, w4, 3, 1, 64, DH_W_L1_0_C2_WT, DH_W_L1_0_C2_B, P2, 1, 1, T4b, 1, 0);
  DH_CONV3("layer1.1.conv1", T4b, nullptr, 64, 0, 0, N2, h4, w4, 3, 1, 64, DH_W_L1_1_C1_WT, DH_W_L1_1_C1_B, nullptr, 0, 1, T4a, 1, 0);
  DH_CONV3("layer1.1.conv2", T4a, nullptr, 64, 0, 0, N2, h4, w4, 3, 1, 64, DH_W_L1_1_C2_WT, DH_W_L1_1_C2_B, T4b, 1, 1, F4, 1, 0);
  float *T8a = ws + p.t8a, *T8b = ws + p.t8b, *T8c = ws + p.t8c, *F8 = ws + p.f8;
  DH_CONV3("layer2.0.conv1", F4, nullptr, 64, 0, 0, N2, h4, w4, 3, 2, 128, DH_W_L2_0_C1_WT, DH_W_L2_0_C1_B, nullptr, 0, 1, T8a, 1, 0);
  DH_CONV3("layer2.0.down", F4, nullptr, 64, 0, 0, N2, h4, w4, 1, 2, 128, DH_W_L2_0_DS_WT, DH_W_L2_0_DS_B, nullptr, 0, 0, T8b, 1, 0);
  DH_CONV3("layer2.0.conv2", T8a, nullptr, 128, 0, 0, N2, h8, w8, 3, 1, 128, DH_W_L2_0_C2_WT, DH_W_L2_0_C2_B, T8b, 1, 1, T8c, 1, 0);
  DH_CONV3("layer2.1.conv1", T8c, nullptr, 128, 0, 0, N2, h8, w8, 3, 1, 128, DH_W_L2_1_C1_WT, DH_W_L2_1_C1_B, nullptr, 0, 1, T8a, 1, 0);
  DH_CONV3("layer2.1.conv2", T8a, nullptr, 128, 0, 0, N2, h8, w8, 3, 1, 128, DH_W_L2_1_C2_WT, DH_W_L2_1_C2_B, T8c, 1, 1, F8, 1, 0);
  float* P8 = ws + p.p8;
  DH_STEP("maxpool_8", 0.0, eb * N2 * 128 * ((double)h8 * w8 + (double)h16 * w16), maxpool(F8, h8, w8, 128, P8));
  float *T16a = ws + p.t16a, *T16b = ws + p.t16b, *T16c = ws + p.t16c, *F16 = ws + p.f16;
  DH_CONV3("layer3.0.conv1", P8, nullptr, 128, 0, 0, N2, h16, w16, 3, 1, 256, DH_W_L3_0_C1_WT, DH_W_L3_0_C1_B, nullptr, 0, 1, T16a, 1, 0);
  DH_CONV3("layer3.0.down", P8, nullptr, 128, 0, 0, N2, h16, w16, 1, 1, 256, DH_W_L3_0_DS_WT, DH_W_L3_0_DS_B, nullptr, 0, 0, T16b, 1, 0);
  DH_CONV3("layer3.0.conv2", T16a, nullptr, 256, 0, 0, N2, h16, w16, 3, 1, 256, DH_W_L3_0_C2_WT, DH_W_L3_0_C2_B, T16b, 1, 1, T16c, 1, 0);
  DH_CONV3("layer3.1.conv1", T16c, nullptr, 256, 0, 0, N2, h16, w16, 3, 1, 256, DH_W_L3_1_C1_WT, DH_W_L3_1_C1_B, nullptr, 0, 1, T16a, 1, 0);
  DH_CONV3("layer3.1.conv2", T16a, nullptr, 256, 0, 0, N2, h16, w16, 3, 1, 256, DH_W_L3_1_C2_WT, DH_W_L3_1_C2_B, T16c, 1, 1, F16, 1, 0);

  // ---- transformer levels 5, 4, 3  (reference networks.py:1297-1318; xBD: model_transformer_encoding.py:385-406)
  float* feats[3] = {F16, F8, F4};
  const int base[3] = {DH_W_LV5_SQ, DH_W_LV4_SQ, DH_W_LV3_SQ};
  static const char* const nm[3][7] = {
      {"squeeze_tok_5", "token_enc_5", "dec_tables_5", "decoder_5_x12", "conv_decode_5", "decoder_5_diff", "conv_layer4"},
      {"squeeze_tok_4", "token_enc_4", "dec_tables_4", "decoder_4_x12", "conv_decode_4", "decoder_4_diff", "conv_layer4"},
      {"squeeze_tok_3", "token_enc_3", "dec_tables_3", "decoder_3_x12", "conv_decode_3", "decoder_3_diff", "conv_layer4"}};
  float* C4 = ws + p.c4;
  const int x3 = (flags & DH_FLAG_DEC_TC_X3) ? 1 : 0;
  // per pixel: x, pos (fp32 weights), out — h16: x and out FP16
  auto dec_bytes_px = [&](const float* pos) { return one ? 32.0 * (2 + 2 + (pos ? 4 : 0)) : 4.0 * 32 * (pos ? 3 : 2); };
  auto level_pre = [&](int i) -> int {
    const Level& L = p.lv[i];
    const int npix = L.h * L.w;
    const float *wtok = Wt(base[i] + 1), *enc = Wt(base[i] + 2), *dec = Wt(base[i] + 3), *pos = Wt(base[i] + 4);
    float *XS = ws + L.xs, *XD = ws + L.xd, *DX = ws + L.dx, *PART = ws + L.part, *MEM = ws + L.mem, *TAB = ws + L.tab;
    const double inner = 64.0 * L.heads;
    const double dec_fl_px = L.depth * 2.0 * (32 * inner + 4 * inner + 4 * inner + inner * 32 + 2 * 32 * 32);
    const double dec_by_px = dec_bytes_px(pos);
    const bool levir = variant == DH_VARIANT_LEVIR;
    {   // squeeze 1x1 + ReLU + tokenizer partials on the tensor cores; xs fp32 for the decoder (LEVIR) / split16 for conv_decode (xBD)
        // (h16: FP16 for both)
      Conv3Args a{};
      a.in0 = feats[i]; a.C0 = L.cin; a.N = N2; a.inH = L.h; a.inW = L.w; a.K = 1; a.stride = 1; a.Cout = 32;
      const size_t plane = (size_t)32 * L.cin;
      a.wt16 = Wt(DH_W_LV5_SQ_WT + i) + 3 * plane; a.wt_plane_bytes = (long long)plane * 4;
      a.out = XS; a.out_split = (levir && !one) ? 0 : 1; a.tok = 1; a.wtok = wtok; a.partials = PART; a.h16 = one;
      DH_STEP(nm[i][0], 2.0 * N2 * npix * 32 * (L.cin + 4 + 4), eb * N2 * npix * (L.cin + 32.0), dh_launch_conv_tc3(a, s));
    }
    const int add_tok_pos = levir ? 1 : (i == 0 ? 1 : 0);
    DH_STEP(nm[i][1], 0.0, 4.0 * N2 * L.nchunk3 * 136.0, dh_launch_token_encoder(PART, B, L.nchunk3, enc, L.heads, add_tok_pos, MEM, s));
    const size_t half = (size_t)B * npix * 32;
    const long long plane2 = (long long)N2 * npix * 32;
    const float* dectc = Wt(DH_W_LV5_DECTC + i);
    if (levir) {
      DH_STEP(nm[i][2], 0.0, 4.0 * 3 * B * L.depth * (double)DH_TABTC_FLOATS, dh_launch_decoder_tables_tc(MEM, B, 0, 3, dec, L.heads, L.depth, TAB, s));
      DH_STEP(nm[i][3], dec_fl_px * N2 * npix, dec_by_px * N2 * npix,
              dh_launch_pixel_decoder_tc(XS, pos, TAB, dectc, N2, L.h, L.w, L.heads, L.depth, nullptr, 1, x3 | (one ? 512 : 256), XD, s));
      DH_CONV3(nm[i][4], XD, reinterpret_cast<float*>(H16(XD) + half), 32, 32, plane2, B, L.h, L.w, 3, 1, 32, DH_W_LV5_DECODE_WT + i, -1,
               nullptr, 0, 0, DX, 0, 0);
    } else {
      DH_STEP(nm[i][2], 0.0, 4.0 * B * L.depth * (double)DH_TABTC_FLOATS, dh_launch_decoder_tables_tc(MEM, B, 2, 1, dec, L.heads, L.depth, TAB, s));
      DH_CONV3(nm[i][4], XS, reinterpret_cast<float*>(H16(XS) + half), 32, 32, plane2, B, L.h, L.w, 3, 1, 32, DH_W_LV5_DECODE_WT + i, -1,
               nullptr, 0, 0, DX, 0, 0);
    }
    return 0;
  };
  auto level_post = [&](int i) -> int {
    const Level& L = p.lv[i];
    const int npix = L.h * L.w;
    const float* pos = Wt(base[i] + 4);
    float *DX = ws + L.dx, *OUT = ws + L.out, *TAB = ws + L.tab;
    const float* skip = (i == 0) ? nullptr : (i == 1 ? ws + p.lv[0].out : C4);     // both fp32 (h16: FP16)
    const int skip_up = (i == 1) ? 2 : 1;
    const double inner = 64.0 * L.heads;
    const double dec_fl_px = L.depth * 2.0 * (32 * inner + 4 * inner + 4 * inner + inner * 32 + 2 * 32 * 32);
    const double dec_by_px = dec_bytes_px(pos);
    const float* dectc = Wt(DH_W_LV5_DECTC + i);
    const float* tab2 = (variant == DH_VARIANT_LEVIR) ? TAB + (size_t)2 * B * L.depth * DH_TABTC_FLOATS : TAB;
    const int out_split = one ? 512 : (i == 0 ? 0 : 256);   // level 5's result is only a decoder skip; levels 4 / 3 feed conv_layer4 / 3
    DH_STEP(nm[i][5], dec_fl_px * B * npix, (dec_by_px + (skip ? 32.0 * eb / (skip_up * skip_up) : 0.0)) * B * npix,
            dh_launch_pixel_decoder_tc(DX, pos, tab2, dectc, B, L.h, L.w, L.heads, L.depth, skip, skip_up, x3 | out_split, OUT, s));
    if (i == 1)   // conv_layer4(up2(out_4)) -> C4 at H/4 (:1335-1336), pixel-shuffle form
      DH_CONV3(nm[i][6], OUT, nullptr, 32, 0, 0, B, L.h, L.w, 3, 1, 128, DH_W_CL4_PSWT, DH_W_CL4_PSB, nullptr, 0, 1, C4, 0, 1);
    return 0;
  };
  AuxStreams* aux = (g_prof.on || (flags & DH_FLAG_SERIAL)) ? nullptr : aux_streams();
  if (aux) {
    if (cudaEventRecord(aux->fork, s_main) != cudaSuccess) return (int)cudaGetLastError();
    for (int i = 1; i <= 2; ++i) {
      s = aux->st[i - 1];
      if (cudaStreamWaitEvent(s, aux->fork, 0) != cudaSuccess) return (int)cudaGetLastError();
      const int rc = level_pre(i);
      if (rc == 0 && cudaEventRecord(aux->join[i - 1], s) != cudaSuccess) { s = s_main; return (int)cudaGetLastError(); }
      s = s_main;
      if (rc != 0) return rc;
    }
  }
  for (int i = 0; i < 3; ++i) {
    int rc = 0;
    if (i == 0 || !aux) rc = level_pre(i);
    else if (cudaStreamWaitEvent(s_main, aux->join[i - 1], 0) != cudaSuccess) rc = (int)cudaGetLastError();
    if (rc == 0) rc = level_post(i);
    if (rc != 0) return rc;
  }
  // ---- UNet head (reference networks.py:1341-1357)
  float *C3 = ws + p.c3, *Y20 = ws + p.y20, *O2 = ws + p.o2, *C2 = ws + p.c2;
  float* OUT3 = ws + p.lv[2].out;                                           // out_3 = level3 + C4 (split16)
  DH_CONV3("conv_layer3", OUT3, nullptr, 32, 0, 0, B, h4, w4, 3, 1, 128, DH_W_CL3_PSWT, DH_W_CL3_PSB, nullptr, 0, 1, C3, 0, 1);
  DH_CONV3("conv_layer2_0.0", F2, F2post, 64, 64, f2_plane, B, h2, w2, 3, 1, 128, DH_W_CL20A_WT, DH_W_CL20A_B, nullptr, 0, 1, Y20, 1, 0);
  DH_CONV3("conv_layer2_0.3", Y20, nullptr, 128, 0, 0, B, h2, w2, 3, 1, 32, DH_W_CL20B_WT, DH_W_CL20B_B, C3, 0, 0, O2, 1, 0);
  DH_CONV3("conv_layer2", O2, nullptr, 32, 0, 0, B, h2, w2, 3, 1, 128, DH_W_CL2_PSWT, DH_W_CL2_PSB, nullptr, 0, 1, C2, 0, 1);
  DH_STEP("classifier", 2.0 * B * H * W * 9 * 32 * output_nc,
          (one ? B * H * W * (2.0 * 32 + 4.0 * output_nc) : 4.0 * B * H * W * (32.0 + output_nc)) + (argmax_u8 ? (double)B * H * W : 0.0),
          one ? dh_launch_classifier_h16(C2, B, H, W, output_nc, Wt(DH_W_CLS_W), Wt(DH_W_CLS_B), logits, argmax_u8, s)
              : dh_launch_classifier(C2, B, H, W, output_nc, Wt(DH_W_CLS_W), Wt(DH_W_CLS_B), logits, argmax_u8, s));
  return 0;
}
}  // namespace


extern "C" int dahitra_forward(const void* const* weights, int n_weights, const float* x1, const float* x2,
                               long long x_batch_stride, float* logits, unsigned char* argmax_u8, void* workspace,
                               size_t workspace_bytes, int variant, int B, int H, int W, int output_nc, int flags,
                               void* stream) {
  DH_REQUIRE(weights && x1 && x2 && logits && workspace, DH_E_NULL);
  DH_REQUIRE(n_weights == DH_W_COUNT, DH_E_WEIGHTS);
  Plan p;
  DH_REQUIRE(variant == DH_VARIANT_LEVIR || variant == DH_VARIANT_XBD, DH_E_VARIANT);
  if (flags & DH_FLAG_ACT_H16) {                // one-FP16-plane storage: the single-pass FP16 convs, the tcgen05 stem and decoder
    constexpr int need = DH_FLAG_CONV_TC | DH_FLAG_TC_MAIN_F16 | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC;
    DH_REQUIRE((flags & need) == need &&
               !(flags & (DH_FLAG_ACT_SPLIT | DH_FLAG_TC_3XTF32 | DH_FLAG_TC_BF16 | DH_FLAG_CONV_TC_V1)), DH_E_VARIANT);
  }
  DH_REQUIRE(make_plan(p, variant, B, H, W, output_nc, flags), DH_E_SHAPE);
  DH_REQUIRE(workspace_bytes >= p.total_floats * sizeof(float), DH_E_WORKSPACE);
  DH_REQUIRE(dh_aligned16(workspace), DH_E_ALIGN);
  for (int i = 0; i < DH_W_COUNT; ++i) {
    const bool optional = (i == DH_W_LV5_POS || i == DH_W_LV4_POS || i == DH_W_LV3_POS);
    DH_REQUIRE(weights[i] || optional, DH_E_WEIGHTS);
    DH_REQUIRE(dh_aligned16(weights[i]), DH_E_ALIGN);
  }
  const cudaStream_t s_main = (cudaStream_t)stream;
  cudaStream_t s = s_main;                      // the stream the launch helpers below use; switched while a level is forked
  float* ws = (float*)workspace;
  dh_set_pdl((flags & DH_FLAG_PDL) ? 1 : 0);
  if (flags & DH_FLAG_ACT_SPLIT) {              // split16 activation storage: needs the FP16 conv operands, the tcgen05 stem and decoder
    constexpr int need = DH_FLAG_CONV_TC | DH_FLAG_TC_MAIN_F16 | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC;
    DH_REQUIRE((flags & need) == need && !(flags & (DH_FLAG_TC_BF16 | DH_FLAG_CONV_TC_V1)), DH_E_VARIANT);
    return forward_split(p, weights, x1, x2, x_batch_stride, logits, argmax_u8, ws, variant, B, H, W, output_nc, flags, s_main);
  }
  if (flags & DH_FLAG_ACT_H16)
    return forward_split(p, weights, x1, x2, x_batch_stride, logits, argmax_u8, ws, variant, B, H, W, output_nc, flags, s_main);
  auto Wt = [&](int slot) { return (const float*)weights[slot]; };
  const int N2 = 2 * B;
  const int h2 = H / 2, w2 = W / 2, h4 = H / 4, w4 = W / 4, h8 = H / 8, w8 = W / 8, h16 = H / 16, w16 = W / 16;

  int conv_flat = 0;                            // ConvArgs::flat of the next conv() calls
  // conv launch + its algorithmic cost (2*MACs as written; one read of the stored inputs/weights, one write)
  auto conv = [&](const char* name, const float* in0, const float* in1, int C0, int C1, int N, int inH, int inW, int up,
                  int K, int stride, int Cout, int wslot, int bslot, const float* res, int relu, float* out) -> int {
    const int wts = wt_slot_of(wslot);
    ConvArgs a{in0, in1, C0, C1, N, inH, inW, up, K, K, stride, K / 2, Cout, Wt(wslot), wts >= 0 ? Wt(wts) : nullptr,
               bslot >= 0 ? Wt(bslot) : nullptr, res, relu, out};
    const int psw = (wslot == DH_W_CL4_W) ? DH_W_CL4_PSWT : (wslot == DH_W_CL3_W) ? DH_W_CL3_PSWT
                  : (wslot == DH_W_CL2_W) ? DH_W_CL2_PSWT : -1;
    a.flat = conv_flat;
    if (up == 2 && psw >= 0 && (flags & DH_FLAG_CONV_TC)) {
      // nearest-x2 upsample + 3x3 conv == 3x3 conv 32 -> 4x32 on the low-res map + pixel-shuffle store
      a.up = 1; a.Cout = 128; a.w = nullptr; a.wt = Wt(psw); a.bias = Wt(psw + 1); a.ps = 1;
    }
    const int rc = conv_dispatch(a, flags, s);
    if (rc != 0) return rc;
    const double OH = (double)(inH * up) / stride, OW = (double)(inW * up) / stride, Cin = C0 + C1;
    const double fl = 2.0 * N * OH * OW * Cout * K * K * Cin;
    const double by = 4.0 * ((double)N * inH * inW * Cin + (double)N * OH * OW * Cout * (res ? 2 : 1) + (double)K * K * Cin * Cout);
    prof_mark(s, name, fl, by);
    return 0;
  };
#define DH_CONV(...)                     \
  do {                                   \
    const int rc__ = conv(__VA_ARGS__);  \
    if (rc__ != 0) return rc__;          \
  } while (0)

  // ---- Siamese trunk on 2B images: [pre batch | post batch]  (reference networks.py:1118-1138, 1323-1324)
  float* F2 = ws + p.f2;
  const double stem_fl = 2.0 * B * h2 * w2 * 64 * 147, stem_by = 4.0 * B * ((double)3 * H * W + (double)h2 * w2 * 64);
  // stem operands: 0 = 1xTF32, 1 = 3xTF32, 2 = folded FP16 (whenever the convolutions run folded: the default mode),
  // 3 = single-pass FP16 (the single-pass 16-bit conv modes; the stem's input is an image, so BF16's range is not needed)
  const int stem_mode = !(flags & DH_FLAG_TC_3XTF32)
                            ? ((flags & (DH_FLAG_TC_MAIN_F16 | DH_FLAG_TC_BF16)) ? 3 : 0)
                            : ((flags & DH_FLAG_TC_FOLD) && (flags & DH_FLAG_TC_MAIN_F16) && (flags & DH_FLAG_TC_X3_BF16)) ? 2 : 1;
  auto stem = [&](const float* xin, float* o) -> int {
    return (flags & DH_FLAG_STEM_TC) ? dh_launch_stem_tc(xin, x_batch_stride, B, H, W, Wt(DH_W_STEM_WTC), Wt(DH_W_STEM_B), o,
                                                         stem_mode, s)
                                     : dh_launch_stem(xin, x_batch_stride, B, H, W, Wt(DH_W_STEM_W), Wt(DH_W_STEM_B), o, s);
  };
  DH_STEP("stem_pre", stem_fl, stem_by, stem(x1, F2));
  DH_STEP("stem_post", stem_fl, stem_by, stem(x2, F2 + (size_t)B * h2 * w2 * 64));
  // conv_layer2_0.0 (the largest launch of the head) needs nothing but the two stem outputs: with DH_FLAG_EARLY_HEAD it is
  // issued now on a lowest-priority side stream, one tile per CTA, so that the hardware scheduler drops its CTAs onto
  // SMs the small token / level-5 / level-4 kernels leave idle; it is joined before conv_layer2_0.3.
  AuxStreams* aux_head = (!g_prof.on && !(flags & DH_FLAG_SERIAL) && (flags & DH_FLAG_EARLY_HEAD) && (flags & DH_FLAG_CONV_TC))
                             ? aux_streams() : nullptr;
  float* Y20 = ws + p.y20;
  if (aux_head) {
    if (cudaEventRecord(aux_head->fork_low, s_main) != cudaSuccess ||
        cudaStreamWaitEvent(aux_head->low, aux_head->fork_low, 0) != cudaSuccess) return (int)cudaGetLastError();
    s = aux_head->low; conv_flat = 1;
    const int rc = conv("conv_layer2_0.0", F2, F2 + (size_t)B * h2 * w2 * 64, 64, 64, B, h2, w2, 1, 3, 1, 128, DH_W_CL20A_W, DH_W_CL20A_B,
                        nullptr, 1, Y20);
    conv_flat = 0;
    const bool ok = rc == 0 && cudaEventRecord(aux_head->join_low, s) == cudaSuccess;
    s = s_main;
    if (!ok) return rc != 0 ? rc : (int)cudaGetLastError();
  }
  float* P2 = ws + p.p2;
  DH_STEP("maxpool_2", 0.0, 4.0 * N2 * 64 * ((double)h2 * w2 + (double)h4 * w4), dh_launch_maxpool(F2, N2, h2, w2, 64, P2, s));
  float *T4a = ws + p.t4a, *T4b = ws + p.t4b, *F4 = ws + p.f4;
  DH_CONV("layer1.0.conv1", P2, nullptr, 64, 0, N2, h4, w4, 1, 3, 1, 64, DH_W_L1_0_C1_W, DH_W_L1_0_C1_B, nullptr, 1, T4a);
  DH_CONV("layer1.0.conv2", T4a, nullptr, 64, 0, N2, h4, w4, 1, 3, 1, 64, DH_W_L1_0_C2_W, DH_W_L1_0_C2_B, P2, 1, T4b);
  DH_CONV("layer1.1.conv1", T4b, nullptr, 64, 0, N2, h4, w4, 1, 3, 1, 64, DH_W_L1_1_C1_W, DH_W_L1_1_C1_B, nullptr, 1, T4a);
  DH_CONV("layer1.1.conv2", T4a, nullptr, 64, 0, N2, h4, w4, 1, 3, 1, 64, DH_W_L1_1_C2_W, DH_W_L1_1_C2_B, T4b, 1, F4);
  float *T8a = ws + p.t8a, *T8b = ws + p.t8b, *T8c = ws + p.t8c, *F8 = ws + p.f8;
  DH_CONV("layer2.0.conv1", F4, nullptr, 64, 0, N2, h4, w4, 1, 3, 2, 128, DH_W_L2_0_C1_W, DH_W_L2_0_C1_B, nullptr, 1, T8a);
  DH_CONV("layer2.0.down", F4, nullptr, 64, 0, N2, h4, w4, 1, 1, 2, 128, DH_W_L2_0_DS_W, DH_W_L2_0_DS_B, nullptr, 0, T8b);
  DH_CONV("layer2.0.conv2", T8a, nullptr, 128, 0, N2, h8, w8, 1, 3, 1, 128, DH_W_L2_0_C2_W, DH_W_L2_0_C2_B, T8b, 1, T8c);
  DH_CONV("layer2.1.conv1", T8c, nullptr, 128, 0, N2, h8, w8, 1, 3, 1, 128, DH_W_L2_1_C1_W, DH_W_L2_1_C1_B, nullptr, 1, T8a);
  DH_CONV("layer2.1.conv2", T8a, nullptr, 128, 0, N2, h8, w8, 1, 3, 1, 128, DH_W_L2_1_C2_W, DH_W_L2_1_C2_B, T8c, 1, F8);
  float* P8 = ws + p.p8;
  DH_STEP("maxpool_8", 0.0, 4.0 * N2 * 128 * ((double)h8 * w8 + (double)h16 * w16), dh_launch_maxpool(F8, N2, h8, w8, 128, P8, s));
  float *T16a = ws + p.t16a, *T16b = ws + p.t16b, *T16c = ws + p.t16c, *F16 = ws + p.f16;
  DH_CONV("layer3.0.conv1", P8, nullptr, 128, 0, N2, h16, w16, 1, 3, 1, 256, DH_W_L3_0_C1_W, DH_W_L3_0_C1_B, nullptr, 1, T16a);
  DH_CONV("layer3.0.down", P8, nullptr, 128, 0, N2, h16, w16, 1, 1, 1, 256, DH_W_L3_0_DS_W, DH_W_L3_0_DS_B, nullptr, 0, T16b);
  DH_CONV("layer3.0.conv2", T16a, nullptr, 256, 0, N2, h16, w16, 1, 3, 1, 256, DH_W_L3_0_C2_W, DH_W_L3_0_C2_B, T16b, 1, T16c);
  DH_CONV("layer3.1.conv1", T16c, nullptr, 256, 0, N2, h16, w16, 1, 3, 1, 256, DH_W_L3_1_C1_W, DH_W_L3_1_C1_B, nullptr, 1, T16a);
  DH_CONV("layer3.1.conv2", T16a, nullptr, 256, 0, N2, h16, w16, 1, 3, 1, 256, DH_W_L3_1_C2_W, DH_W_L3_1_C2_B, T16c, 1, F16);

  // ---- transformer levels 5, 4, 3  (reference networks.py:1297-1318; xBD: model_transformer_encoding.py:385-406)
  const float* feats[3] = {F16, F8, F4};
  const int base[3] = {DH_W_LV5_SQ, DH_W_LV4_SQ, DH_W_LV3_SQ};
  static const char* const nm[3][7] = {
      {"squeeze_tok_5", "token_enc_5", "dec_tables_5", "decoder_5_x12", "conv_decode_5", "decoder_5_diff", "conv_layer4"},
      {"squeeze_tok_4", "token_enc_4", "dec_tables_4", "decoder_4_x12", "conv_decode_4", "decoder_4_diff", "conv_layer4"},
      {"squeeze_tok_3", "token_enc_3", "dec_tables_3", "decoder_3_x12", "conv_decode_3", "decoder_3_diff", "conv_layer4"}};
  float* C4 = ws + p.c4;
  // level_pre(i): everything of level i that depends only on the trunk; level_post(i): the part that needs the level above
  auto level_pre = [&](int i) -> int {
    const Level& L = p.lv[i];
    const int npix = L.h * L.w;
    const float *wsq = Wt(base[i] + 0), *wtok = Wt(base[i] + 1), *enc = Wt(base[i] + 2), *dec = Wt(base[i] + 3),
                *pos = Wt(base[i] + 4);
    float *XS = ws + L.xs, *XD = ws + L.xd, *DX = ws + L.dx, *PART = ws + L.part, *MEM = ws + L.mem, *TAB = ws + L.tab;
    // as-written FLOPs per pixel of one decoder call (help_funcs.py:66-114): q proj + dots + attn.V + out proj + MLP
    const double inner = 64.0 * L.heads;
    const double dec_fl_px = L.depth * 2.0 * (32 * inner + 4 * inner + 4 * inner + inner * 32 + 2 * 32 * 32);
    const double dec_by_px = 4.0 * 32 * (pos ? 3 : 2);
    DH_STEP(nm[i][0], 2.0 * N2 * npix * 32 * (L.cin + 4 + 4), 4.0 * N2 * npix * (L.cin + 32.0),
            dh_launch_squeeze_tokens(feats[i], N2, npix, L.cin, wsq, wtok, XS, PART, s));
    const int add_tok_pos = (variant == DH_VARIANT_LEVIR) ? 1 : (i == 0 ? 1 : 0);
    DH_STEP(nm[i][1], 0.0, 4.0 * N2 * L.nchunk * 136.0, dh_launch_token_encoder(PART, B, L.nchunk, enc, L.heads, add_tok_pos, MEM, s));
    const size_t half = (size_t)B * npix * 32;
    // decoder launches: CUDA-core kernels, or the tcgen05 pair (DH_FLAG_DEC_TC) with its own table layout
    const bool dtc = (flags & DH_FLAG_DEC_TC) != 0;
    const float* dectc = Wt(DH_W_LV5_DECTC + i);
    const size_t tabf = dtc ? (size_t)DH_TABTC_FLOATS : (size_t)DH_TAB_FLOATS(L.heads);
    auto tables = [&](int first, int ncalls) -> int {
      return dtc ? dh_launch_decoder_tables_tc(MEM, B, first, ncalls, dec, L.heads, L.depth, TAB, s)
                 : dh_launch_decoder_tables(MEM, B, first, ncalls, dec, L.heads, L.depth, TAB, s);
    };
    if (variant == DH_VARIANT_LEVIR) {
      DH_STEP(nm[i][2], 0.0, 4.0 * 3 * B * L.depth * tabf, tables(0, 3));
      DH_STEP(nm[i][3], dec_fl_px * N2 * npix, dec_by_px * N2 * npix,
              (dtc ? dh_launch_pixel_decoder_tc(XS, pos, TAB, dectc, N2, L.h, L.w, L.heads, L.depth, nullptr, 1,
                                                (flags & DH_FLAG_DEC_TC_X3) ? 1 : 0, XD, s)
                   : dh_launch_pixel_decoder(XS, pos, TAB, dec, N2, L.h, L.w, L.heads, L.depth, nullptr, 1, XD, s)));
      DH_CONV(nm[i][4], XD, XD + half, 32, 32, B, L.h, L.w, 1, 3, 1, 32, base[i] + 5, -1, nullptr, 0, DX);
    } else {
      DH_STEP(nm[i][2], 0.0, 4.0 * B * L.depth * tabf, tables(2, 1));
      DH_CONV(nm[i][4], XS, XS + half, 32, 32, B, L.h, L.w, 1, 3, 1, 32, base[i] + 5, -1, nullptr, 0, DX);
    }
    return 0;
  };
  auto level_post = [&](int i) -> int {
    const Level& L = p.lv[i];
    const int npix = L.h * L.w;
    const float *dec = Wt(base[i] + 3), *pos = Wt(base[i] + 4);
    float *DX = ws + L.dx, *OUT = ws + L.out, *TAB = ws + L.tab;
    // what the reference adds to this level's result: nothing (level 5), up2(out_5) (level 4, :1333),
    // conv_layer4(up2(out_4)) at the same resolution (level 3, :1340)
    const float* skip = (i == 0) ? nullptr : (i == 1 ? ws + p.lv[0].out : C4);
    const int skip_up = (i == 1) ? 2 : 1;
    const double inner = 64.0 * L.heads;
    const double dec_fl_px = L.depth * 2.0 * (32 * inner + 4 * inner + 4 * inner + inner * 32 + 2 * 32 * 32);
    const double dec_by_px = 4.0 * 32 * (pos ? 3 : 2);
    const bool dtc = (flags & DH_FLAG_DEC_TC) != 0;
    const float* dectc = Wt(DH_W_LV5_DECTC + i);
    const size_t tabf = dtc ? (size_t)DH_TABTC_FLOATS : (size_t)DH_TAB_FLOATS(L.heads);
    const float* tab2 = (variant == DH_VARIANT_LEVIR) ? TAB + (size_t)2 * B * L.depth * tabf : TAB;
    DH_STEP(nm[i][5], dec_fl_px * B * npix, (dec_by_px + (skip ? 128.0 / (skip_up * skip_up) : 0.0)) * B * npix,
            (dtc ? dh_launch_pixel_decoder_tc(DX, pos, tab2, dectc, B, L.h, L.w, L.heads, L.depth, skip, skip_up,
                                              (flags & DH_FLAG_DEC_TC_X3) ? 1 : 0, OUT, s)
                 : dh_launch_pixel_decoder(DX, pos, tab2, dec, B, L.h, L.w, L.heads, L.depth, skip, skip_up, OUT, s)));
    if (i == 1)   // conv_layer4(up2(out_4)) -> C4 at H/4 (:1335-1336)
      DH_CONV(nm[i][6], OUT, nullptr, 32, 0, B, L.h, L.w, 2, 3, 1, 32, DH_W_CL4_W, DH_W_CL4_B, nullptr, 1, C4);
    return 0;
  };
  // fork levels 4 and 3 unless profiling (per-launch events want one stream) or DH_FLAG_SERIAL asks for one stream
  AuxStreams* aux = (g_prof.on || (flags & DH_FLAG_SERIAL)) ? nullptr : aux_streams();
  if (aux) {
    if (cudaEventRecord(aux->fork, s_main) != cudaSuccess) return (int)cudaGetLastError();
    for (int i = 1; i <= 2; ++i) {
      s = aux->st[i - 1];
      if (cudaStreamWaitEvent(s, aux->fork, 0) != cudaSuccess) return (int)cudaGetLastError();
      const int rc = level_pre(i);
      if (rc == 0 && cudaEventRecord(aux->join[i - 1], s) != cudaSuccess) { s = s_main; return (int)cudaGetLastError(); }
      s = s_main;
      if (rc != 0) return rc;
    }
  }
  for (int i = 0; i < 3; ++i) {
    int rc = 0;
    if (i == 0 || !aux) rc = level_pre(i);
    else if (cudaStreamWaitEvent(s_main, aux->join[i - 1], 0) != cudaSuccess) rc = (int)cudaGetLastError();
    if (rc == 0) rc = level_post(i);
    if (rc != 0) return rc;
  }
  // ---- UNet head (reference networks.py:1341-1357)
  float *C3 = ws + p.c3, *O2 = ws + p.o2, *C2 = ws + p.c2;
  const float* OUT3 = ws + p.lv[2].out;                                   // out_3 = level3 + C4
  DH_CONV("conv_layer3", OUT3, nullptr, 32, 0, B, h4, w4, 2, 3, 1, 32, DH_W_CL3_W, DH_W_CL3_B, nullptr, 1, C3);   // on up2(out_3)
  const float* A128 = F2;
  const float* B128 = F2 + (size_t)B * h2 * w2 * 64;
  if (aux_head) {
    if (cudaStreamWaitEvent(s_main, aux_head->join_low, 0) != cudaSuccess) return (int)cudaGetLastError();
  } else {
    DH_CONV("conv_layer2_0.0", A128, B128, 64, 64, B, h2, w2, 1, 3, 1, 128, DH_W_CL20A_W, DH_W_CL20A_B, nullptr, 1, Y20);  // conv+BN+ReLU
  }
  DH_CONV("conv_layer2_0.3", Y20, nullptr, 128, 0, B, h2, w2, 1, 3, 1, 32, DH_W_CL20B_W, DH_W_CL20B_B, C3, 0, O2);       // + out_3
  DH_CONV("conv_layer2", O2, nullptr, 32, 0, B, h2, w2, 2, 3, 1, 32, DH_W_CL2_W, DH_W_CL2_B, nullptr, 1, C2);            // on up2(out_2)
  DH_STEP("classifier", 2.0 * B * H * W * 9 * 32 * output_nc, 4.0 * B * H * W * (32.0 + output_nc) + (argmax_u8 ? (double)B * H * W : 0.0),
          dh_launch_classifier(C2, B, H, W, output_nc, Wt(DH_W_CLS_W), Wt(DH_W_CLS_B), logits, argmax_u8, s));
  return 0;
}

// Diagnostic twin of dahitra_forward: records a CUDA event after every launch, SYNCHRONISES the stream, and
// returns per-launch device time plus the algorithmic FLOPs / bytes of each launch.  Not for the hot path.
//   ms/flops/bytes: host arrays of capacity `cap`; names: host array of `cap` const char*; returns the number
//   of launches (>0) or an error code (<=0).
extern "C" int dahitra_forward_profiled(const void* const* weights, int n_weights, const float* x1, const float* x2,
                                        long long x_batch_stride, float* logits, unsigned char* argmax_u8,
                                        void* workspace, size_t workspace_bytes, int variant, int B, int H, int W,
                                        int output_nc, int flags, void* stream, int cap, float* ms, double* flops,
                                        double* bytes, const char** names) {
  DH_REQUIRE(ms && flops && bytes && names && cap > 0, DH_E_NULL);
  cudaStream_t s = (cudaStream_t)stream;
  if (!g_prof.created) {
    for (int i = 0; i <= PROF_MAX; ++i)
      if (cudaEventCreate(&g_prof.ev[i]) != cudaSuccess) return -(int)cudaGetLastError() - 1000;
    g_prof.created = true;
  }
  g_prof.n = 0;
  g_prof.on = true;
  cudaEventRecord(g_prof.ev[0], s);
  const int rc = dahitra_forward(weights, n_weights, x1, x2, x_batch_stride, logits, argmax_u8, workspace, workspace_bytes,
                                 variant, B, H, W, output_nc, flags, stream);
  g_prof.on = false;
  if (rc != 0) return rc > 0 ? -rc - 1000 : rc;
  const cudaError_t e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return -(int)e - 1000;
  const int n = g_prof.n < cap ? g_prof.n : cap;
  for (int i = 0; i < n; ++i) {
    cudaEventElapsedTime(&ms[i], g_prof.ev[i], g_prof.ev[i + 1]);
    flops[i] = g_prof.rec[i].flops;
    bytes[i] = g_prof.rec[i].bytes;
    names[i] = g_prof.rec[i].name;
  }
  return n;
}
