"""Native inference engine: host-side weight preparation + the call into ``dahitra_forward``.

Weight preparation (once per set of weights, re-done after ``load_state_dict`` / ``train()`` / ``.to()``):
  * eval-mode BatchNorm folded into the preceding convolution (W' = W*g/sigma, b' = beta - mu*g/sigma)
  * conv weights re-laid-out OIHW -> [KH*KW*Cin][Cout] (implicit-GEMM "B" operand, Cout contiguous)
  * token encoder / pixel decoder products collapsed to per-head 32x32 matrices in fp64
    (Mqk = dim^-0.5 Wq^T Wk, Mov = Wo Wv), second LayerNorm of each decoder layer folded into W1/b1
  * decoder positional embeddings NCHW -> [h*w][32]
Layouts are documented slot by slot in include/dahitra_b200.h.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _lib

BN_EPS = 1e-5
SCALE = 32 ** -0.5
LEVELS = ((5, 256, 4, 4), (4, 128, 4, 4), (3, 64, 8, 8))   # (k, trunk channels, heads, decoder depth)

DH_VARIANT_LEVIR, DH_VARIANT_XBD = 0, 1
DH_FLAG_CONV_TC, DH_FLAG_TC_3XTF32, DH_FLAG_TC_STRIDE2, DH_FLAG_DEC_TC, DH_FLAG_STEM_TC, DH_FLAG_DEC_TC_X3 = 1, 2, 4, 8, 16, 32
DH_FLAG_CONV_TC_V1, DH_FLAG_CONV_TC_2CTA, DH_FLAG_SERIAL, DH_FLAG_TC_X3_BF16, DH_FLAG_TC_BF16 = 64, 128, 256, 512, 1024
DH_FLAG_TC_MAIN_F16, DH_FLAG_TC_FOLD, DH_FLAG_EARLY_HEAD, DH_FLAG_ACT_SPLIT, DH_FLAG_PDL = 2048, 4096, 8192, 16384, 32768
DH_FLAG_ACT_H16 = 65536
MODES = {
    "fp32": 0,                                             # every contraction in fp32 FMA (strict)
    "fp32_tcdec": DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3,      # strict + the 3xTF32 (fp32-grade) tensor-core decoder
    # fp32-grade accuracy on the tensor cores: every product is error-compensated (three partial products, fp32
    # accumulation).  Convolutions: main product in FP16 (11-bit significand like TF32, 16-bit operands), the two
    # correction products in BF16 (fp32 exponent range) — half the tensor-core cycles of three TF32 products and a
    # slightly smaller error.  Operands beyond the FP16 range (|v| > 65504, or < 1e-7) fall back on the BF16 terms
    # (bf16-grade accuracy for those values only).  The 7x7 stem runs the same way; pixel decoder: 3xTF32.
    # The f16(a).r_w correction shares its A operand with the main product, so both come out of ONE N-doubled FP16 MMA
    # on the filter tile [f16(w) ; f16(2^11 r_w)] and are added in the epilogue (DH_FLAG_TC_FOLD).
    # Activations that feed a convolution are STORED as the pair the MMAs consume — hi = f16(a), lo = f16(2^11 (a - hi)), the
    # same 4 bytes per element as fp32 (DH_FLAG_ACT_SPLIT, csrc/conv_tc3.cu): a.w = h_a.h_w + 2^-11 (h_a.l_w + l_a.h_w), all
    # three products on FP16 MMAs, TMA lands the operands directly, and the tokenizer's 1x1 squeeze runs on the tensor cores.
    "tf32x3": DH_FLAG_CONV_TC | DH_FLAG_TC_3XTF32 | DH_FLAG_TC_X3_BF16 | DH_FLAG_TC_MAIN_F16 | DH_FLAG_TC_FOLD | DH_FLAG_TC_STRIDE2
              | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3 | DH_FLAG_ACT_SPLIT | DH_FLAG_PDL,
    # ... with fp32 activation storage and an in-kernel splitter pass (round 1's default; f16 main + bf16 remainders)
    "tf32x3_fp32act": DH_FLAG_CONV_TC | DH_FLAG_TC_3XTF32 | DH_FLAG_TC_X3_BF16 | DH_FLAG_TC_MAIN_F16 | DH_FLAG_TC_FOLD | DH_FLAG_TC_STRIDE2
                      | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3,
    # ... with three separate products per (tap, chunk) and the 3xTF32 stem (~10 % slower)
    "tf32x3_unfolded": DH_FLAG_CONV_TC | DH_FLAG_TC_3XTF32 | DH_FLAG_TC_X3_BF16 | DH_FLAG_TC_MAIN_F16 | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC
                       | DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3,
    # the same with the main product in TF32 (no range caveat, ~15 % slower)
    "tf32x3_tf32main": DH_FLAG_CONV_TC | DH_FLAG_TC_3XTF32 | DH_FLAG_TC_X3_BF16 | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC
                       | DH_FLAG_DEC_TC_X3,
    "tf32x3_pure": DH_FLAG_CONV_TC | DH_FLAG_TC_3XTF32 | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3,
    "tf32": DH_FLAG_CONV_TC | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3,
    # single-pass FP16 operands in the convolutions (TF32-grade significand, half the operand bytes of "tf32";
    # saturating outside +-65504) and in the stem, 3xTF32 decoder
    "f16": DH_FLAG_CONV_TC | DH_FLAG_TC_MAIN_F16 | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3,
    # reduced precision: BF16 operands in every convolution (fp32 storage / accumulation), single-pass FP16 stem (its input is an
    # image), 3xTF32 decoder
    "bf16": DH_FLAG_CONV_TC | DH_FLAG_TC_BF16 | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3,
    # reduced precision, half the activation bytes: "f16" operands AND every workspace tensor stored as one FP16 plane (2 bytes
    # per element, saturating at +-65504; tokenizer partials / token memories / decoder tables stay fp32), single-pass FP16
    # convolutions (conv_tc3.cu single-plane form), 3xTF32 decoder
    "h16": DH_FLAG_CONV_TC | DH_FLAG_TC_MAIN_F16 | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC | DH_FLAG_DEC_TC_X3
           | DH_FLAG_ACT_H16 | DH_FLAG_PDL,
    "tf32_fast": DH_FLAG_CONV_TC | DH_FLAG_TC_STRIDE2 | DH_FLAG_STEM_TC | DH_FLAG_DEC_TC,   # 1xTF32 decoder too
}

# fp32-grade accuracy on arbitrary checkpoints at tensor-core speed; "fp32" is the strict CUDA-core mode
DEFAULT_MODE = "tf32x3"


def resolve_mode(mode):
    if isinstance(mode, int):
        return mode
    if mode not in MODES:
        raise ValueError(f"dahitra_b200: unknown precision mode {mode!r}; choose from {sorted(MODES)}")
    return MODES[mode]


def slot_names():
    lib = _lib.load()
    out, i = [], 0
    while True:
        s = lib.dahitra_weight_slot_name(i)
        if s is None:
            return out
        out.append(s.decode())
        i += 1


# ----------------------------------------------------------------------------- host-side preparation
def _fold_conv_bn(sd, conv, bn):
    w = sd[conv + ".weight"].double()
    if bn is None:
        return w, (sd[conv + ".bias"].double() if (conv + ".bias") in sd else None)
    g, b = sd[bn + ".weight"].double(), sd[bn + ".bias"].double()
    mu, var = sd[bn + ".running_mean"].double(), sd[bn + ".running_var"].double()
    k = g / torch.sqrt(var + BN_EPS)
    return w * k[:, None, None, None], b - mu * k


def _khwc(w):
    """OIHW -> [KH*KW*Cin][Cout]"""
    o, i, kh, kw = w.shape
    return w.permute(2, 3, 1, 0).reshape(kh * kw * i, o)


def upsample_phase_filter(w, b):
    """nn.Upsample(x2, nearest) followed by a 3x3 pad-1 conv == four 2x2 convs on the low-res map, one per
    output-pixel phase (py, px): rows r of the 3x3 filter that land on the same low-res row are summed.
    out[2i+py, 2j+px] = sum_{u,v in {-1,0,1}} W3[(py,px)][u,v] . x[i+u, j+v]  with
        py = 0: u=-1 <- r=0 ; u=0 <- r=1,2        py = 1: u=0 <- r=0,1 ; u=+1 <- r=2      (same for columns)
    Returns the K-major filter [4*Cout][9*Cin] (row = phase*Cout + co, col = (u+1)*3*Cin + (v+1)*Cin + ci) and
    the bias repeated per phase.  w: (Cout, Cin, 3, 3) float64."""
    cout, cin = w.shape[:2]
    rows = {0: {-1: [0], 0: [1, 2]}, 1: {0: [0, 1], 1: [2]}}
    W3 = torch.zeros(4, cout, 3, 3, cin, dtype=w.dtype)
    for py in (0, 1):
        for px in (0, 1):
            for u, rs in rows[py].items():
                for v, ss in rows[px].items():
                    acc = torch.zeros(cout, cin, dtype=w.dtype)
                    for r in rs:
                        for s in ss:
                            acc += w[:, :, r, s]
                    W3[py * 2 + px, :, u + 1, v + 1, :] = acc
    return W3.reshape(4 * cout, 9 * cin), b.repeat(4)


def tf32_round(x):
    """nearest TF32-representable value (10 explicit mantissa bits; ties away from zero like cvt.rna.tf32.f32)"""
    b = x.to(torch.float32).contiguous().view(torch.int32)
    return ((b + 0x1000) & ~0x1FFF).view(torch.float32)


def tf32_split(x):
    """x (float64) -> (hi, lo) float64 with hi, lo exactly representable in TF32 and hi + lo = x to ~2^-22 relative."""
    hi = tf32_round(x).double()
    lo = tf32_round(x - hi).double()
    return hi, lo


def kmajor_split(wt):
    """K-major filter [Cout][K] (float64) -> float32 [5][Cout][K]:
      plane 0  TF32-rounded values (B_hi; all the 1xTF32 kernels read)
      plane 1  their TF32-rounded remainders (B_lo of the 3xTF32 kernels)
      plane 2  raw bits of a bf16 [2][Cout][K] array: bf16(w) and bf16(w - B_hi), the filter operands of the two
               correction products when they run as BF16 MMAs (DH_FLAG_TC_X3_BF16)."""
    wt = wt.contiguous().double()
    hi, lo = tf32_split(wt)
    b16 = torch.stack([wt, wt - hi]).to(torch.float32).to(torch.bfloat16).contiguous()       # [2][Cout][K] bf16
    packed = b16.view(torch.int16).reshape(-1).view(torch.float32).reshape(wt.shape)          # same bytes as [Cout][K] fp32
    # plane 3: f16(w) (saturated to the f16 range) and bf16(w - f16(w)) for the FP16-main-product mode
    h16 = wt.clamp(-65504.0, 65504.0).to(torch.float32).to(torch.float16)
    r16 = (wt - h16.double()).to(torch.float32).to(torch.bfloat16)
    packed_f = torch.cat([h16.contiguous().view(torch.int16).reshape(-1), r16.contiguous().view(torch.int16).reshape(-1)]) \
        .view(torch.float32).reshape(wt.shape)
    # plane 4: f16(2^11 (w - f16(w))) (the remainder scaled into the normal f16 range; second half unused) for the
    # folded-correction mode
    s16 = ((wt - h16.double()) * 2048.0).clamp(-65504.0, 65504.0).to(torch.float32).to(torch.float16)
    packed_s = torch.cat([s16.contiguous().view(torch.int16).reshape(-1), torch.zeros(s16.numel(), dtype=torch.int16)]) \
        .view(torch.float32).reshape(wt.shape)
    return torch.cat([torch.stack([hi, lo]).to(torch.float32), packed[None], packed_f[None], packed_s[None]])


def stem_tc_image(w147):
    """[147][64] stem filter, K ordered (r, s, ci) like DH_W_STEM_W -> the tcgen05 stem's B operands (float32 buffer):
    K re-ordered to (ci, r, s8) — 21 groups of 8 (a zero + 7 taps) padded to 192 — then
      [0, 24576)       TF32 [hi | lo] images of 6 K-step tiles of the swizzled B[n=co][k 32]   (1xTF32 / 3xTF32 stem)
      [24576, 36864)   raw bits of the folded FP16 image: 3 K-step tiles of 128 rows x 64 k 16-bit, rows 0..63 = f16(w),
                       rows 64..127 = f16(2^11 (w - f16(w)))
      [36864, 43008)   raw bits of 3 K-step tiles of 64 rows x 64 k bf16(w)                    (folded FP16 stem)"""
    w = w147.double().reshape(7, 7, 3, 64)                                   # [r][s][ci][co]
    wk = torch.zeros(24, 8, 64, dtype=torch.float64)
    wk[:21, 1:8] = w.permute(2, 0, 1, 3).reshape(21, 7, 64)                  # group = ci*7 + r; slot 0 = the alignment pad
    wk = wk.reshape(192, 64)
    hi, lo = tf32_split(wk)
    img = lambda m: torch.cat([swizzle128(m[kt * 32:(kt + 1) * 32].T.contiguous()) for kt in range(6)])
    h16 = wk.clamp(-65504.0, 65504.0).to(torch.float32).to(torch.float16)
    s16 = ((wk - h16.double()) * 2048.0).clamp(-65504.0, 65504.0).to(torch.float32).to(torch.float16)
    main = torch.cat([h16, s16], dim=1).view(torch.int16)                    # [192][128]: f16 w | scaled remainder
    corr = wk.to(torch.float32).to(torch.bfloat16).view(torch.int16)         # [192][64]
    img16 = lambda m: torch.cat([swizzle128_16(m[kt * 64:(kt + 1) * 64].T.contiguous()) for kt in range(3)]).view(torch.float32)
    return torch.cat([img(hi).to(torch.float32), img(lo).to(torch.float32), img16(main), img16(corr)])


def swizzle128_16(m):
    """[rows][64] matrix of 16-bit values B[n][k] -> flat K-major SWIZZLE_128B image (rows of 128 B, the 16-byte chunk
    index XOR-ed with row % 8): element (n, k) lands at n*64 + (((k>>3) ^ (n&7)) << 3 | (k&7))."""
    rows = m.shape[0]
    n = torch.arange(rows)[:, None].expand(rows, 64)
    k = torch.arange(64)[None, :].expand(rows, 64)
    idx = n * 64 + ((((k >> 3) ^ (n & 7)) << 3) | (k & 7))
    out = torch.empty(rows * 64, dtype=m.dtype)
    out[idx.reshape(-1)] = m.reshape(-1)
    return out


def swizzle128(m):
    """[rows][32] matrix B[n][k] -> flat K-major SWIZZLE_128B shared-memory image (rows of 128 B, the 16-byte
    chunk index XOR-ed with row % 8): element (n, k) lands at n*32 + (((k>>2) ^ (n&7)) << 2 | (k&3))."""
    rows = m.shape[0]
    n = torch.arange(rows)[:, None].expand(rows, 32)
    k = torch.arange(32)[None, :].expand(rows, 32)
    idx = n * 32 + ((((k >> 2) ^ (n & 7)) << 2) | (k & 3))
    out = torch.empty(rows * 32, dtype=m.dtype)
    out[idx.reshape(-1)] = m.reshape(-1)
    return out


def _heads(w, h):                       # (h*64, 32) -> (h, 64, 32)
    return w.reshape(h, -1, w.shape[-1])


def prepare_weights(sd: dict, variant: int, out_nc: int) -> dict:
    """state_dict (reference key layout, any device/dtype) -> {slot name: fp32 CPU tensor (or None)}."""
    sd = {k: v.detach().cpu() for k, v in sd.items()}
    P = {}

    tc_slots = {"DH_W_L1_0_C1", "DH_W_L1_0_C2", "DH_W_L1_1_C1", "DH_W_L1_1_C2", "DH_W_L2_0_C2", "DH_W_L2_1_C1",
                "DH_W_L2_1_C2", "DH_W_L3_0_C1", "DH_W_L3_0_C2", "DH_W_L3_0_DS", "DH_W_L3_1_C1", "DH_W_L3_1_C2",
                "DH_W_CL20A", "DH_W_CL20B", "DH_W_L2_0_C1", "DH_W_L2_0_DS"}

    def put_conv(slot, conv, bn):
        w, b = _fold_conv_bn(sd, conv, bn)
        P[slot + "_W"] = _khwc(w)
        P[slot + "_B"] = b
        if slot in tc_slots:
            P[slot + "_WT"] = kmajor_split(_khwc(w).T)           # [2][Cout][KH*KW*Cin]: K-major B operand, TF32 hi / lo

    put_conv("DH_W_STEM", "resnet.conv1", "resnet.bn1")
    P["DH_W_STEM_WTC"] = stem_tc_image(P["DH_W_STEM_W"])
    for li in (1, 2, 3):
        for bi in (0, 1):
            p = f"resnet.layer{li}.{bi}"
            put_conv(f"DH_W_L{li}_{bi}_C1", p + ".conv1", p + ".bn1")
            put_conv(f"DH_W_L{li}_{bi}_C2", p + ".conv2", p + ".bn2")
            if (p + ".downsample.0.weight") in sd:
                put_conv(f"DH_W_L{li}_{bi}_DS", p + ".downsample.0", p + ".downsample.1")
    for k, cin, heads, depth in LEVELS:
        s = f"DH_W_LV{k}_"
        P[s + "SQ"] = sd[f"conv_squeeze_{k}.0.weight"].double()[:, :, 0, 0].T          # [Cin][32]
        P[s + "TOK"] = sd[f"conv_token_{k}.weight"].double()[:, :, 0, 0].T             # [32][4]
        P[s + "SQ_WT"] = kmajor_split(P[s + "SQ"].T)                                   # [32][Cin] K-major planes (conv_tc3 tok launch)
        P[s + "DECODE"] = _khwc(sd[f"conv_decode_{k}.weight"].double())
        P[s + "DECODE_WT"] = kmajor_split(P[s + "DECODE"].T)
        # ---- token encoder pack
        t = f"transformer_{k}.layers.0"
        if variant == DH_VARIANT_LEVIR:
            pos = sd[f"pos_embedding_{k}"].double().reshape(-1) if f"pos_embedding_{k}" in sd \
                else torch.zeros(256, dtype=torch.float64)
        else:   # xBD: only the H/16 level adds one, and it is pos_embedding_3 (model_transformer_encoding.py:358-366)
            pos = sd["pos_embedding_3"].double().reshape(-1) if (k == 5 and "pos_embedding_3" in sd) \
                else torch.zeros(256, dtype=torch.float64)      # with_pos=None builds no token embeddings (reference default)
        wqkv = sd[t + ".0.fn.fn.to_qkv.weight"].double()
        inner = heads * 64
        wq, wk, wv = (_heads(wqkv[i * inner:(i + 1) * inner], heads) for i in range(3))
        wo = sd[t + ".0.fn.fn.to_out.0.weight"].double().reshape(32, heads, 64).permute(1, 0, 2)   # (h, c, d)
        mqk = SCALE * torch.einsum("hdc,hde->hce", wq, wk)              # [h][c][c']
        mvoT = torch.einsum("hcd,hde->hec", wo, wv)                     # [h][c'][c]
        P[s + "ENC"] = torch.cat([
            pos, sd[t + ".0.fn.norm.weight"].double(), sd[t + ".0.fn.norm.bias"].double(),
            mqk.reshape(-1), mvoT.reshape(-1), sd[t + ".0.fn.fn.to_out.0.bias"].double(),
            sd[t + ".1.fn.norm.weight"].double(), sd[t + ".1.fn.norm.bias"].double(),
            sd[t + ".1.fn.fn.net.0.weight"].double().T.reshape(-1), sd[t + ".1.fn.fn.net.0.bias"].double(),
            sd[t + ".1.fn.fn.net.3.weight"].double().T.reshape(-1), sd[t + ".1.fn.fn.net.3.bias"].double()])
        # ---- pixel decoder pack
        layers = []
        for l in range(depth):
            d = f"transformer_decoder_{k}.layers.{l}"
            wq = _heads(sd[d + ".0.fn.fn.to_q.weight"].double(), heads)
            wk = _heads(sd[d + ".0.fn.fn.to_k.weight"].double(), heads)
            wv = _heads(sd[d + ".0.fn.fn.to_v.weight"].double(), heads)
            wo = sd[d + ".0.fn.fn.to_out.0.weight"].double().reshape(32, heads, 64).permute(1, 0, 2)
            mqkT = SCALE * torch.einsum("hdc,hde->hec", wq, wk)         # [h][c'][c]
            movT = torch.einsum("hcd,hde->hec", wo, wv)                 # [h][c'][c]
            g2, b2n = sd[d + ".1.fn.norm.weight"].double(), sd[d + ".1.fn.norm.bias"].double()
            w1, b1 = sd[d + ".1.fn.fn.net.0.weight"].double(), sd[d + ".1.fn.fn.net.0.bias"].double()
            w2, b2 = sd[d + ".1.fn.fn.net.3.weight"].double(), sd[d + ".1.fn.fn.net.3.bias"].double()
            layers += [sd[d + ".0.fn.norm.weight"].double(), sd[d + ".0.fn.norm.bias"].double(),
                       mqkT.reshape(-1), movT.reshape(-1), sd[d + ".0.fn.fn.to_out.0.bias"].double(),
                       (w1 * g2[None, :]).T.reshape(-1), b1 + w1 @ b2n, w2.T.reshape(-1), b2]
        P[s + "DEC"] = torch.cat(layers)
        # ---- tensor-core decoder pack: pre-swizzled B operands + cumulative biases (include/dahitra_b200.h)
        tc_layers, cum = [], torch.zeros(32, dtype=torch.float64)
        for l in range(depth):
            d = f"transformer_decoder_{k}.layers.{l}"
            g2, b2n = sd[d + ".1.fn.norm.weight"].double(), sd[d + ".1.fn.norm.bias"].double()
            w1, b1 = sd[d + ".1.fn.fn.net.0.weight"].double(), sd[d + ".1.fn.fn.net.0.bias"].double()
            w2, b2 = sd[d + ".1.fn.fn.net.3.weight"].double(), sd[d + ".1.fn.fn.net.3.bias"].double()
            cba = cum + sd[d + ".0.fn.fn.to_out.0.bias"].double()
            cum = cba + b2
            w1h, w1l = tf32_split(w1 * g2[None, :])
            w2h, w2l = tf32_split(w2)
            tc_layers += [swizzle128(w1h), swizzle128(w2h), b1 + w1 @ b2n, cba, cum.clone(), swizzle128(w1l), swizzle128(w2l)]
        P[s + "DECTC"] = torch.cat(tc_layers)
        # ---- decoder positional embedding
        if variant == DH_VARIANT_LEVIR:
            pe = sd.get(f"pos_embedding_decoder_{k}")
        else:
            pe = sd.get("pos_embedding_decoder_3") if k == 5 else None
        P[s + "POS"] = None if pe is None else pe.double()[0].permute(1, 2, 0).reshape(-1, 32)
    for name, key in (("DH_W_CL4", "conv_layer4.0"), ("DH_W_CL3", "conv_layer3.0"), ("DH_W_CL2", "conv_layer2.0")):
        put_conv(name, key, None)
        pw, pb = upsample_phase_filter(sd[key + ".weight"].double(), sd[key + ".bias"].double())
        P[name + "_PSWT"], P[name + "_PSB"] = kmajor_split(pw), pb
    put_conv("DH_W_CL20A", "conv_layer2_0.0", "conv_layer2_0.1")
    put_conv("DH_W_CL20B", "conv_layer2_0.3", None)
    wc = sd["classifier.weight"].double()
    assert wc.shape[0] == out_nc
    P["DH_W_CLS_W"] = wc.permute(2, 3, 0, 1).reshape(9, out_nc, 32)
    P["DH_W_CLS_B"] = sd["classifier.bias"].double()
    return {k: (None if v is None else v.to(torch.float32).contiguous()) for k, v in P.items()}


def prepare_weights_c(sd: dict, variant: int, out_nc: int):
    """The same preparation through the C ABI (`dahitra_prepare_weights`, csrc/prepare.cu — host code, no PyTorch inside):
    -> (flat fp32 CPU tensor holding every slot, list of float offsets per slot, -1 = absent).  What a C / C++ consumer of
    the library runs; engine.prepare_weights above is the executable specification it is tested against."""
    lib = _lib.load()
    keep, recs = [], []
    for k, v in sd.items():
        if not torch.is_tensor(v) or not v.dtype.is_floating_point or v.dim() > 4:
            continue
        t = v.detach().cpu().contiguous()
        if t.dtype not in (torch.float32, torch.float64):
            t = t.float()
        keep.append((k.encode(), t))
    arr = (_lib.DhTensor * len(keep))()
    for i, (name, t) in enumerate(keep):
        arr[i].name, arr[i].data = name, t.data_ptr()
        arr[i].dtype, arr[i].ndim = (0 if t.dtype == torch.float32 else 1), t.dim()
        for j, d in enumerate(t.shape):
            arr[i].shape[j] = d
    n = lib.dahitra_prepare_weights(arr, len(keep), variant, out_nc, None, 0, None)
    if n <= 0:
        _lib.check(int(n), "dahitra_prepare_weights")
    flat = torch.zeros(n, dtype=torch.float32)
    offs = (C.c_longlong * len(slot_names()))()
    n2 = lib.dahitra_prepare_weights(arr, len(keep), variant, out_nc, flat.data_ptr(), n, offs)
    if n2 != n:
        _lib.check(int(n2) if n2 < 0 else -6, "dahitra_prepare_weights")
    return flat, list(offs)


F16_MAX = 65504.0


def _filter_absmax(flat: torch.Tensor, offs: dict):
    """largest |w| over the folded fp32 filters of a prepared buffer (the `_W` / `_DECODE` / `_SQ` slots: every convolution's
    BatchNorm-folded weights) and the slot that holds it; NaN if any of them is not finite"""
    import bisect
    ends = sorted(offs.values()) + [flat.numel()]
    worst, where = 0.0, None
    for name, o in offs.items():
        if name.endswith(("_W", "_DECODE", "_SQ")):
            seg = flat[o:ends[bisect.bisect_right(ends, o)]]
            m = float(seg.abs().max()) if seg.numel() else 0.0
            if not m <= worst:                  # larger, or NaN
                worst, where = m, name
                if m != m:
                    break
    return worst, where


class PreparedWeights:
    """Device copy of the prepared slots + the C pointer table handed to dahitra_forward.

    The preparation itself runs in the library (`dahitra_prepare_weights`, csrc/prepare.cu: plain host C++, what a consumer
    without PyTorch runs); DAHITRA_PREPARE=py selects the Python specification above instead (bit-identical slots,
    tests/test_host_cpu.py)."""

    def __init__(self, sd, variant, out_nc, device):
        names = slot_names()
        if os.environ.get("DAHITRA_PREPARE", "c") == "py":
            host = prepare_weights(sd, variant, out_nc)
            missing = [n for n in names if n not in host]
            if missing:
                raise RuntimeError(f"weight preparation does not produce slots {missing}")
            offs, total = {}, 0                     # one flat buffer, every slot 256-byte aligned
            for n in names:
                if host[n] is not None:
                    offs[n] = total
                    total += (host[n].numel() + 63) // 64 * 64
            flat = torch.zeros(total, dtype=torch.float32)
            for n, o in offs.items():
                flat[o:o + host[n].numel()] = host[n].reshape(-1)
        else:
            flat, off_list = prepare_weights_c(sd, variant, out_nc)
            offs = {n: o for n, o in zip(names, off_list) if o >= 0}
        self.filter_absmax = _filter_absmax(flat, offs)     # (value, slot) over the folded fp32 filters, checked on the host
        if not (self.filter_absmax[0] <= F16_MAX):            # also true for NaN
            import warnings
            warnings.warn(f"dahitra_b200: folded filter {self.filter_absmax[1]} has max |w| = {self.filter_absmax[0]:.4g}, outside the FP16 "
                          "operand range of the default mode (values saturate at 65504); use net.set_mode('tf32x3_tf32main') or 'fp32' "
                          "for this checkpoint (DESIGN.md, 'FP16 operand caveat')", RuntimeWarning, stacklevel=3)
        self.flat = flat.to(device)
        base = self.flat.data_ptr()
        self.table = (C.c_void_p * len(names))(*[(base + 4 * offs[n]) if n in offs else None for n in names])
        self.n = len(names)
        self.names = names
        self.offs = offs
        # positions each decoder positional-embedding slot covers (the forward checks them against the input size)
        self.pos_positions = {}
        for k in (5, 4, 3):
            key = f"pos_embedding_decoder_{k}" if variant == DH_VARIANT_LEVIR else ("pos_embedding_decoder_3" if k == 5 else None)
            if key is not None and key in sd and f"DH_W_LV{k}_POS" in offs:
                self.pos_positions[f"DH_W_LV{k}_POS"] = int(sd[key].shape[2] * sd[key].shape[3])

    def ptr(self, name):
        return self.flat.data_ptr() + 4 * self.offs[name] if name in self.offs else None


# ----------------------------------------------------------------------------- engine
class NativeEngine:
    def __init__(self):
        self._preps = {}            # (device, variant) -> PreparedWeights; all dropped when the live tensors change
        self._tensors = None        # the module's parameters + buffers (cached walk of the module tree)
        self._fingerprint = None
        self._ws = {}               # (device, stream, variant, B, H, W, nc) -> workspace; released only explicitly
        # precision mode: DAHITRA_FLAGS (raw DH_FLAG_* bitmask) > DAHITRA_MODE (a MODES name) > DEFAULT_MODE
        if "DAHITRA_FLAGS" in os.environ:
            self.flags = int(os.environ["DAHITRA_FLAGS"])
        else:
            self.flags = resolve_mode(os.environ.get("DAHITRA_MODE", DEFAULT_MODE))
        self.last_argmax = None

    # an engine holds device pointers (ctypes table) and scratch memory: copies / pickles of the owning module get a fresh,
    # empty engine that carries only the precision mode (copy.deepcopy(net) for EMA / SWA, torch.save(net))
    def __deepcopy__(self, memo):
        e = NativeEngine.__new__(NativeEngine)
        e.__setstate__(self.__getstate__())
        return e

    def __getstate__(self):
        return {"flags": self.flags}

    def __setstate__(self, st):
        self._preps, self._tensors, self._fingerprint, self._ws, self.last_argmax = {}, None, None, {}, None
        self.flags = st.get("flags", MODES[DEFAULT_MODE])

    def set_mode(self, mode):
        """mode: a key of MODES or a raw DH_FLAG_* bitmask.  Every mode runs from the same prepared weights, so switching
        back and forth does not rebuild or re-upload anything."""
        self.flags = resolve_mode(mode)

    @property
    def mode(self):
        return next((k for k, v in MODES.items() if v == self.flags), f"flags{self.flags}")

    def invalidate(self):
        """Forget the prepared weights AND the cached list of the module's tensors (call after replacing a Parameter
        object; in-place updates, load_state_dict, .to() and optimizer steps are detected without it)."""
        self._preps = {}
        self._tensors = None
        self._fingerprint = None

    def release_workspaces(self):
        """Free the scratch buffers (one per (device, stream, shape)).  Never done implicitly: a captured CUDA graph keeps
        pointing at the workspace it was captured with."""
        self._ws = {}

    def _live_fingerprint(self, module):
        # cheap staleness check on every forward (~25 us): the version counter of every parameter / buffer changes on any
        # in-place write (optimizer.step, copy_, load_state_dict on this module or on a parent, EMA updates), the storage
        # address on .to() / .cuda()
        ts = self._tensors
        if ts is None:
            ts = self._tensors = [t for t in list(module.parameters()) + list(module.buffers())]
        return (tuple(t._version for t in ts), ts[0].data_ptr() if ts else 0, len(ts))

    def _prepared(self, module, device):
        fp = self._live_fingerprint(module)
        if fp != self._fingerprint:
            self._preps = {}
            self._fingerprint = fp
        key = (str(device), module.VARIANT)
        prep = self._preps.get(key)
        if prep is None:
            variant = DH_VARIANT_LEVIR if module.VARIANT == "levir" else DH_VARIANT_XBD
            prep = self._preps[key] = PreparedWeights(module.state_dict(), variant, module.output_nc, device)
        return prep

    def _workspace(self, lib, device, variant, B, H, W, nc):
        stream = torch.cuda.current_stream(device)
        capturing = torch.cuda.is_current_stream_capturing()
        # one workspace per stream: two forwards issued on different streams must not share scratch memory.  A workspace
        # first needed while a graph is being captured is allocated from that graph's pool and is never handed to eager
        # launches (key "capture"); entries are only freed by release_workspaces().
        nbytes = lib.dahitra_workspace_bytes(variant, B, H, W, nc, self.flags)      # depends on the flags (buffer reuse plan)
        if nbytes == 0:
            raise RuntimeError(f"dahitra_b200: unsupported shape B={B} H={H} W={W} (H, W must be multiples of 32)")
        key = (str(device), "capture" if capturing else stream.cuda_stream, variant, B, H, W, nc, nbytes)
        ws = self._ws.get(key)
        if ws is None:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=device)
            self._ws[key] = ws
        return ws

    def run(self, module, x1, x2, batch_stride, B, H, W, want_argmax=False):
        lib = _lib.load()
        dev = x1.device
        variant = DH_VARIANT_LEVIR if module.VARIANT == "levir" else DH_VARIANT_XBD
        prep = self._prepared(module, dev)
        for name, hw in module.pos_shapes(H, W).items():
            have = prep.pos_positions.get(name)
            if have is not None and have != hw:
                raise RuntimeError(
                    f"dahitra_b200: decoder positional embedding {name} has {have} positions but the input needs {hw} "
                    f"(the {module.VARIANT} variant only runs at the resolution its embeddings were built for, like the reference)")
        nc = module.output_nc
        ws = self._workspace(lib, dev, variant, B, H, W, nc)
        logits = torch.empty((B, nc, H, W), dtype=torch.float32, device=dev)
        amax = torch.empty((B, H, W), dtype=torch.uint8, device=dev) if want_argmax else None
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):        # the library sizes grids / creates its side streams on the CURRENT device
            rc = lib.dahitra_forward(prep.table, prep.n, x1.data_ptr(), x2.data_ptr(), batch_stride,
                                     logits.data_ptr(), amax.data_ptr() if amax is not None else None,
                                     ws.data_ptr(), ws.numel(), variant, B, H, W, nc, self.flags, stream)
        _lib.check(rc, "dahitra_forward")
        self.last_argmax = amax
        return logits

    def profile_pair(self, module, x1, x2):
        """One forward with a CUDA event after every launch (synchronises).  -> list of
        {name, ms, flops, bytes} in launch order; diagnostic only (bench.py roofline)."""
        lib = _lib.load()
        x1 = x1.float().contiguous()
        x2 = x2.float().contiguous()
        B, _, H, W = x1.shape
        dev = x1.device
        variant = DH_VARIANT_LEVIR if module.VARIANT == "levir" else DH_VARIANT_XBD
        prep = self._prepared(module, dev)
        nc = module.output_nc
        ws = self._workspace(lib, dev, variant, B, H, W, nc)
        logits = torch.empty((B, nc, H, W), dtype=torch.float32, device=dev)
        cap = 160
        ms, fl, by = (C.c_float * cap)(), (C.c_double * cap)(), (C.c_double * cap)()
        names = (C.c_char_p * cap)()
        stream = torch.cuda.current_stream(dev).cuda_stream
        with torch.cuda.device(dev):
            n = lib.dahitra_forward_profiled(prep.table, prep.n, x1.data_ptr(), x2.data_ptr(), 3 * H * W, logits.data_ptr(),
                                             None, ws.data_ptr(), ws.numel(), variant, B, H, W, nc, self.flags, stream,
                                             cap, ms, fl, by, names)
        if n <= 0:
            _lib.check(n if n > -1000 else -(n + 1000), "dahitra_forward_profiled")
        return [dict(name=names[i].decode(), ms=float(ms[i]), flops=float(fl[i]), bytes=float(by[i])) for i in range(n)]

    def forward_pair(self, module, x1, x2, want_argmax=False):
        if x1.shape != x2.shape or x1.dim() != 4 or x1.shape[1] != 3:
            raise RuntimeError(f"dahitra_b200: expected two (B,3,H,W) tensors, got {tuple(x1.shape)} and {tuple(x2.shape)}")
        x1 = x1.float().contiguous()
        x2 = x2.float().contiguous()
        B, _, H, W = x1.shape
        return self.run(module, x1, x2, 3 * H * W, B, H, W, want_argmax)

    def forward_stacked(self, module, x, want_argmax=False):
        """xBD calling convention: x = cat[pre, post] on channels, (B,6,H,W)."""
        if x.dim() != 4 or x.shape[1] != 6:
            raise RuntimeError(f"dahitra_b200: expected a (B,6,H,W) tensor, got {tuple(x.shape)}")
        x = x.float().contiguous()
        B, _, H, W = x.shape
        return self.run(module, x, x[:, 3:], 6 * H * W, B, H, W, want_argmax)
