"""GPU: the h16 mode (every workspace activation stored as one FP16 plane, DH_FLAG_ACT_H16).

Block tests feed operands that are exactly FP16-representable, so every product is exact in fp32; a result must then be the
fp64 result rounded to FP16 within 1 ulp of that rounding (plus 1e-6 of the sum of |a.w| for results near zero, where the
fp32 accumulation order dominates).  Whole-forward tests use the bar tests/test_gpu_forward.py::test_tensor_core_modes
states for the reduced-precision mode."""
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import abi
import emulate as E
from oracle import dahitra_oracle as O
from oracle import synth
from test_oracle_golden import Args

pytestmark = pytest.mark.gpu
DEV = "cuda"
H16_BIT = 128                                          # dahitra_conv2d_split: storage bit of the h16 format


def q16(*shape, seed=0, scale=1.0):
    """random values that are exactly representable in FP16 (fp32 tensor on the device)"""
    return (torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale).half().float().to(DEV)


def ulp16(v):
    """spacing of FP16 at |v| (fp64): 2^(e - 11) for |v| in [2^(e-1), 2^e), 2^-24 in the subnormal range"""
    _, e = torch.frexp(v.abs().double().clamp_min(2.0 ** -14))
    return torch.ldexp(torch.ones_like(v, dtype=torch.float64), e - 11)


def assert_within_ulp(y, ref, mag, what):
    """y: FP16 result; ref: fp64 result; mag: fp64 sum of |a.w| per element"""
    y, ref, mag = y.double().cpu(), ref.double().cpu(), mag.double().cpu()
    r16 = ref.half().double()
    d = (y - r16).abs()
    bad = d > ulp16(r16) + 1e-6 * mag
    print(f"[h16] {what}: max|d|={float(d.max()):.3e} >1ulp:{int((d > ulp16(r16)).sum())} bad:{int(bad.sum())}/{d.numel()}")
    assert not bad.any(), f"{what}: {int(bad.sum())} elements beyond 1 FP16 ulp (max|d| {float(d.max()):.3e})"


def conv_h16(in0, in1, wt, bias, res, relu, K, stride, mode=0, wtok=None, sched=0, out_fp16=True):
    """dahitra_conv2d_split with the h16 bit: in0 / in1 / res FP16 NHWC planes; wt: the conv's *_WT image [5][Cout][K]"""
    from dahitra_b200 import _lib
    lib = _lib.load()
    N, inH, inW, C0 = in0.shape
    C1 = 0 if in1 is None else in1.shape[-1]
    Cout = wt.shape[1]
    OH, OW = inH // stride, inW // stride
    shape = (N, 2 * OH, 2 * OW, 32) if mode == 1 else (N, OH, OW, Cout)
    out = torch.empty(shape, device=DEV, dtype=torch.float16 if out_fp16 else torch.float32)
    parts = None
    if mode == 2:
        parts = torch.empty((N, ((inH + 15) // 16) * ((inW + 7) // 8), 4, 34), device=DEV, dtype=torch.float32)
    p = lambda t: None if t is None else t.data_ptr()
    rc = lib.dahitra_conv2d_split(p(in0), p(in1), C0, C1, 0, 0, N, inH, inW, K, stride, Cout, p(wt), p(bias), p(res), int(res is not None),
                                  int(relu), p(out), int(out_fp16), mode | sched | H16_BIT, p(wtok), p(parts),
                                  torch.cuda.current_stream().cuda_stream)
    return rc, out, parts


def kmajor(w_kc):
    from dahitra_b200.engine import kmajor_split
    return kmajor_split(w_kc.detach().cpu().double()).float().contiguous().to(DEV)


H16_CONVS = [  # (N, H, W, C0, C1, Cout, K, stride, res, relu, bias)
    (2, 16, 16, 32, 0, 32, 1, 1, False, False, False),        # one chunk, one tap
    (2, 32, 32, 64, 0, 64, 3, 1, True, True, True),           # layer1 conv2 (+identity, ReLU)
    (2, 32, 32, 128, 0, 128, 3, 1, True, True, True),         # layer2
    (1, 64, 64, 64, 0, 128, 3, 2, False, True, True),         # layer2.0.conv1: stride 2 (four phase halos)
    (2, 32, 32, 64, 0, 128, 1, 2, False, False, True),        # layer2.0 downsample (1x1 stride 2)
    (2, 16, 16, 128, 0, 256, 1, 1, False, False, True),       # layer3.0 downsample (two N tiles)
    (1, 16, 16, 256, 0, 256, 3, 1, True, True, True),         # layer3 (72 (tap, chunk) steps)
    (2, 32, 32, 32, 32, 32, 3, 1, False, False, False),       # conv_decode on a virtual concat
    (1, 64, 64, 64, 64, 128, 3, 1, False, True, True),        # conv_layer2_0.0 (concat, C1 > 0)
    (1, 64, 64, 128, 0, 32, 3, 1, True, False, True),         # conv_layer2_0.3 + out_3 (FP16 residual)
    (1, 20, 28, 32, 0, 64, 3, 1, True, True, True),           # ragged edges
    (3, 36, 20, 64, 0, 32, 3, 2, False, False, True),         # ragged + stride 2
    (40, 64, 64, 64, 0, 64, 3, 1, True, True, True),          # 1280 tiles: filter resident, every CTA walks many tiles
]


@pytest.mark.parametrize("cfg", H16_CONVS)
def test_conv_h16(cfg):
    """conv_tc3 single-plane form vs fp64 of the same FP16 values, rounded to FP16; resident and streamed filter identical"""
    N, H, W, C0, C1, Cout, K, stride, res, relu, bias = cfg
    x0 = q16(N, H, W, C0, seed=1)
    x1 = q16(N, H, W, C1, seed=2) if C1 else None
    Kt = K * K * (C0 + C1)
    w = q16(Kt, Cout, seed=3, scale=Kt ** -0.5)
    b = q16(Cout, seed=4) if bias else None
    OH, OW = H // stride, W // stride
    r = q16(N, OH, OW, Cout, seed=5) if res else None
    wt = kmajor(w.t())
    h = lambda t: None if t is None else t.half().contiguous()
    rc, y, _ = conv_h16(h(x0), h(x1), wt, b, h(r), relu, K, stride)
    assert rc == 0, rc
    rc, ys, _ = conv_h16(h(x0), h(x1), wt, b, h(r), relu, K, stride, sched=64)      # filter streamed from L2
    assert rc == 0, rc
    torch.cuda.synchronize()
    assert torch.equal(y, ys), "resident and streamed filter differ"
    xc = (x0 if x1 is None else torch.cat([x0, x1], -1)).double().cpu()
    ref = E.conv_nhwc(xc, w.double().cpu(), None if b is None else b.double().cpu(), K, stride, K // 2,
                      None if r is None else r.double().cpu(), relu, 1)
    mag = E.conv_nhwc(xc.abs(), w.double().cpu().abs(), None, K, stride, K // 2, None, False, 1)
    assert_within_ulp(y, ref, mag, str(cfg))
    if cfg == H16_CONVS[1]:                 # fp32 output from FP16 operands (out_split = 0)
        rc, yf, _ = conv_h16(h(x0), h(x1), wt, b, h(r), relu, K, stride, out_fp16=False)
        assert rc == 0
        torch.cuda.synchronize()
        assert float((yf.double().cpu() - ref).abs().max()) <= 1e-5 * float(ref.abs().max())


def test_conv_h16_pixel_shuffle():
    """nearest-x2 upsample + 3x3 conv (conv_layer4/3/2) on one FP16 plane, pixel-shuffle store of one FP16 plane"""
    from dahitra_b200.engine import upsample_phase_filter
    for (N, H, W) in [(2, 16, 16), (1, 24, 40), (12, 64, 64)]:
        x = q16(N, H, W, 32, seed=1)
        g = torch.Generator().manual_seed(2)
        w = (torch.randn(32, 32, 3, 3, generator=g) * (288 ** -0.5)).half().double()
        b = torch.randn(32, generator=g).half().double()
        wt, pb = upsample_phase_filter(w, b)                   # sums of up to 4 taps: exact in fp32, may round in FP16
        from dahitra_b200.engine import kmajor_split
        wtk = kmajor_split(wt).float().contiguous().to(DEV)
        xu = x.double().cpu().permute(0, 3, 1, 2).repeat_interleave(2, 2).repeat_interleave(2, 3)
        ref = F.relu(F.conv2d(xu, w, b, 1, 1)).permute(0, 2, 3, 1)
        mag = F.conv2d(xu.abs(), w.abs(), None, 1, 1).permute(0, 2, 3, 1)
        outs = []
        for sched in (0, 64):
            rc, y, _ = conv_h16(x.half(), None, wtk, pb.float().to(DEV), None, True, 3, 1, mode=1, sched=sched)
            assert rc == 0, rc
            outs.append(y)
        torch.cuda.synchronize()
        assert torch.equal(outs[0], outs[1])
        # the phase filter holds sums of up to four FP16 taps, which FP16 may not represent: compare with the fp64 statement of
        # what the kernel multiplies (the filter rounded to FP16 as the engine stores it)
        wt16 = wt.half().double()
        phases = F.conv2d(x.double().cpu().permute(0, 3, 1, 2), wt16.view(128, 3, 3, 32).permute(0, 3, 1, 2),
                          pb.float().double(), 1, 1).relu()
        ref16 = torch.empty(N, 2 * H, 2 * W, 32, dtype=torch.float64)
        for j in range(4):
            ref16[:, j >> 1::2, j & 1::2, :] = phases[:, 32 * j:32 * (j + 1)].permute(0, 2, 3, 1)
        assert_within_ulp(y, ref16, mag, f"pixel shuffle {N}x{H}x{W}")
        d = (y.double().cpu() - ref).abs()
        assert float(d.max()) <= 2e-2 * float(ref.abs().max())          # and close to the unrounded upsample conv


def test_conv_h16_tokenizer():
    """conv_tc3 tok epilogue in the single-plane form: xs as one FP16 plane, softmax partials fp32, vs fp64"""
    for (N, H, W, Cin) in [(2, 16, 16, 256), (2, 64, 64, 64), (1, 24, 40, 64)]:
        feat = q16(N, H, W, Cin, seed=1)
        wsq = q16(Cin, 32, seed=2, scale=Cin ** -0.5)
        wtok = rnd32(32, 4, seed=3)
        rc, xs, parts = conv_h16(feat.half(), None, kmajor(wsq.t()), None, None, False, 1, 1, mode=2, wtok=wtok)
        assert rc == 0, rc
        torch.cuda.synchronize()
        fq = feat.double().cpu().reshape(N, H * W, Cin)
        xr = torch.relu(fq @ wsq.double().cpu())
        mag = fq.abs() @ wsq.double().cpu().abs()
        assert_within_ulp(xs.reshape(N, H * W, 32), xr, mag, f"tok xs {N}x{H}x{W}x{Cin}")
        p = parts.double().cpu()
        M = p[..., 0].max(dim=1, keepdim=True).values
        sc = torch.exp(p[..., 0] - M)
        tok = (p[..., 2:] * sc[..., None]).sum(1) / (p[..., 1] * sc).sum(1)[..., None]
        a = torch.softmax(torch.einsum("npc,cl->nlp", xr, wtok.double().cpu()), dim=-1)
        ref = torch.einsum("nlp,npc->nlc", a, xr)
        assert float((tok - ref).abs().max()) <= 1e-4 * float(ref.abs().max())


def rnd32(*shape, seed=0, scale=1.0):
    return (torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale).to(DEV)


def test_conv_h16_rejects_cta_pairs():
    x = q16(2, 32, 32, 64, seed=1).half()
    wt = kmajor(q16(576, 128, seed=2).t())
    rc, _, _ = conv_h16(x, None, wt, None, None, False, 3, 1, sched=32)
    assert rc == -5                                          # DH_E_VARIANT: no CTA-pair variant, and no silent fall-back
    rc, _, _ = conv_h16(x, None, wt, None, None, False, 3, 1, sched=16)
    assert rc == 0


@pytest.mark.parametrize("shape", [(2, 16, 16, 64), (1, 20, 28, 128), (3, 64, 64, 64)])
def test_maxpool_h16(shape):
    from dahitra_b200 import _lib
    N, H, W, C = shape
    x = rnd32(N, H, W, C, seed=3, scale=4.0).half()
    out = torch.empty(N, H // 2, W // 2, C, device=DEV, dtype=torch.float16)
    _lib.check(_lib.load().dahitra_maxpool3x3s2_h16(x.data_ptr(), N, H, W, C, out.data_ptr(), torch.cuda.current_stream().cuda_stream))
    ref = F.max_pool2d(x.permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1)
    assert torch.equal(out, ref)


@pytest.mark.parametrize("shape", [(2, 64, 64), (1, 96, 160), (1, 40, 72)])
def test_stem_h16(shape):
    """single-pass FP16 stem with one FP16 output plane vs the fp64 stem of the FP16-rounded input and filter"""
    from dahitra_b200 import _lib
    from dahitra_b200.engine import stem_tc_image
    N, H, W = shape
    x = q16(N, 3, H, W, seed=1)
    w = q16(147, 64, seed=2, scale=147 ** -0.5)
    b = rnd32(64, seed=3)
    wtc = stem_tc_image(w.cpu()).float().to(DEV)
    out = torch.empty(N, H // 2, W // 2, 64, device=DEV, dtype=torch.float16)
    _lib.check(_lib.load().dahitra_stem_tc(x.data_ptr(), 3 * H * W, N, H, W, wtc.data_ptr(), b.data_ptr(), out.data_ptr(), 3 | 512,
                                           torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    ref = E.stem(x.double(), w.double(), b.double())
    mag = E.stem(x.double().abs(), w.double().abs(), torch.zeros_like(b).double()).cpu() + b.double().abs().cpu()
    assert_within_ulp(out, ref, mag, f"stem {shape}")


@pytest.mark.parametrize("k,h,w", [(5, 16, 16), (4, 32, 32), (3, 24, 40)])
def test_pixel_decoder_h16(k, h, w, levir_template):
    """FP16 x / skip / out against the fp32-input decoder on the same (upcast) values, its output rounded to FP16"""
    from dahitra_b200.engine import prepare_weights
    sd = dict(synth.synth_state_dict(levir_template, seed=3, style="default"))
    heads, depth = O.LEVELS[k]["heads"], O.LEVELS[k]["depth"]
    sd[f"pos_embedding_decoder_{k}"] = torch.randn(1, 32, h, w, generator=torch.Generator().manual_seed(5))
    P = {n: (None if v is None else v.to(DEV)) for n, v in prepare_weights(sd, 0, 2).items()}
    B = 2
    x = q16(B, h * w, 32, seed=8)
    mem = rnd32(B, 3, 4, 32, seed=9)
    s = f"DH_W_LV{k}_"
    tab = abi.decoder_tables_tc(mem, 0, 1, P[s + "DEC"], heads, depth)
    for skip_up in (0, 1, 2):
        sk = None if skip_up == 0 else q16(B, h // skip_up, w // skip_up, 32, seed=11)
        su = max(skip_up, 1)
        ref = abi.pixel_decoder_tc(x, P[s + "POS"], tab, P[s + "DECTC"], h, w, heads, depth, sk, su, x3=1)
        y = torch.empty(B, h * w, 32, device=DEV, dtype=torch.float16)
        from dahitra_b200 import _lib
        p = lambda t: None if t is None else t.data_ptr()
        x16, sk16 = x.half(), (None if sk is None else sk.half())        # kept alive until the launch has run
        _lib.check(_lib.load().dahitra_pixel_decoder_tc(x16.data_ptr(), p(P[s + "POS"]), tab.data_ptr(), P[s + "DECTC"].data_ptr(),
                                                        B, h, w, heads, depth, p(sk16), su, 1 | 512,
                                                        y.data_ptr(), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        r16 = ref.double().cpu().half().double()
        d = (y.double().cpu() - r16).abs()
        assert bool((d <= ulp16(r16)).all()), f"skip_up {skip_up}: max|d| {float(d.max()):.3e}"


@pytest.mark.parametrize("nc", [2, 5])
def test_classifier_h16(nc):
    from dahitra_b200 import _lib
    x = q16(2, 48, 80, 32, seed=1)
    w = rnd32(9, nc, 32, seed=2, scale=0.1)
    b = rnd32(nc, seed=3, scale=0.1)
    N, H, W, _ = x.shape
    logits = torch.empty(N, nc, H, W, device=DEV)
    am = torch.empty(N, H, W, device=DEV, dtype=torch.uint8)
    x16 = x.half()                                             # kept alive until the launch has run
    _lib.check(_lib.load().dahitra_classifier_h16(x16.data_ptr(), N, H, W, nc, w.data_ptr(), b.data_ptr(), logits.data_ptr(),
                                                  am.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    wt = w.reshape(3, 3, nc, 32).permute(2, 3, 0, 1).double()
    ref = F.conv2d(x.double().permute(0, 3, 1, 2), wt, b.double(), 1, 1)
    d = (logits.double() - ref).abs()
    assert bool((d <= 1e-5 * ref.abs() + 1e-6 * float(ref.abs().max())).all()), float(d.max())
    assert torch.equal(am.long(), logits.argmax(1))


# ------------------------------------------------------------------------------------------------ whole forward
def make_net(sd, nc=2):
    from dahitra_b200.networks import BASE_Transformer_UNet
    net = BASE_Transformer_UNet(3, nc, 'learned', resnet_stages_num=4, with_decoder_pos='learned', enc_depth=1, dec_depth=8)
    net.load_state_dict(sd, strict=True)
    return net.to(DEV).eval()


def eager_tf32(net, *xs):
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    with torch.no_grad():
        net.train(False)
        y = net._forward_autograd(*xs).double().cpu()
    torch.backends.cuda.matmul.allow_tf32 = False
    return y


def reduced_precision_bar(y, ref, weights, what, yt=None):
    """test_tensor_core_modes' bar for the reduced-precision mode; the strict north-star tolerance is reported, not asserted"""
    d = (y - ref).abs()
    agree = float((y.argmax(1) == ref.argmax(1)).float().mean())
    strict_ok = bool((d <= 1e-4 + 1e-3 * ref.abs()).all())
    extra = ""
    if yt is not None:
        extra = f" | eager-PyTorch-TF32 mean|d|={float((yt - ref).abs().mean()):.3e}"
    print(f"[parity] h16 {what} ({weights}): max|d|={float(d.max()):.3e} mean|d|={float(d.mean()):.3e} "
          f"ref_absmax={float(ref.abs().max()):.3e} argmax_agree={agree:.6f} strict-north-star-met={strict_ok}{extra}")
    if weights == "defineG":
        assert int((d > 2e-3 + 2e-2 * ref.abs()).sum()) == 0 and agree >= 0.995
    else:
        assert float(d.mean()) <= 5.0 * float((yt - ref).abs().mean()) + 1e-5 and agree >= 0.99


@pytest.mark.parametrize("weights", ["defineG", "default"])
def test_h16_levir_vs_oracle(weights, levir_template):
    from dahitra_b200.networks import define_G
    from dahitra_b200.engine import MODES
    if weights == "defineG":
        torch.manual_seed(0)
        net = define_G(Args(), gpu_ids=[0]).eval()
        sd = {k: v.cpu() for k, v in net.state_dict().items()}
    else:
        sd = synth.synth_state_dict(levir_template, seed=3, style="default")
        net = make_net(sd)
    net.set_mode("h16")
    assert net._engine.flags == MODES["h16"] and net._engine.mode == "h16"
    x1, x2 = synth.synth_pair(2, 256, 256, seed=2, kind="uniform")
    with torch.no_grad():
        y = net(x1.to(DEV), x2.to(DEV)).double().cpu()
    ref = O.forward_levir(sd, x1, x2, dtype=torch.float64)
    reduced_precision_bar(y, ref, weights, "LEVIR 256", eager_tf32(net, x1.to(DEV), x2.to(DEV)))


@pytest.mark.parametrize("weights", ["normal", "default"])
def test_config5_tiled1024_h16_vs_oracle(weights, levir_template):
    """configs[4]: one uint8 1024x1024 pair, tiled to 16 x 256x256 on the device, LEVIR module with output_nc=5, h16 mode"""
    from dahitra_b200.networks import BASE_Transformer_UNet, init_weights
    from dahitra_b200.inputs import normalize_u8
    net = BASE_Transformer_UNet(3, 5, 'learned', resnet_stages_num=4, with_decoder_pos='learned', enc_depth=1, dec_depth=8)
    if weights == "normal":
        torch.manual_seed(0)
        init_weights(net, 'normal', 0.02)
    else:
        net.load_state_dict(synth.synth_state_dict(net.state_dict(), seed=3, style="default"))
    net = net.to(DEV).eval().set_mode("h16")
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    g = torch.Generator(device=DEV).manual_seed(7)
    pre = torch.randint(0, 256, (1, 1024, 1024, 3), device=DEV, generator=g, dtype=torch.uint8)
    post = torch.randint(0, 256, (1, 1024, 1024, 3), device=DEV, generator=g, dtype=torch.uint8)
    t1, t2 = normalize_u8(pre, "levir", tile=256), normalize_u8(post, "levir", tile=256)
    assert t1.shape == (16, 3, 256, 256)
    with torch.no_grad():
        y = net(t1, t2).double().cpu()
    ref = O.forward_levir(sd, t1.cpu(), t2.cpu(), dtype=torch.float64)
    reduced_precision_bar(y, ref, "defineG" if weights == "normal" else "default", "configs[4] tiled 1024",
                          None if weights == "normal" else eager_tf32(net, t1, t2))


def test_h16_xbd_1024_golden(golden_dir):
    """xBD 1024x1024, 5 classes, in h16 against the fp64 reference values of the golden fixture (every 8th pixel)"""
    from dahitra_b200.xbd import BASE_Transformer_UNet as X
    g = np.load(os.path.join(golden_dir, "xbd_synth6_1024.npz"))
    net = X(input_nc=3, output_nc=5, token_len=4, resnet_stages_num=4, with_pos="learned", with_decoder_pos="learned",
            enc_depth=1, dec_depth=8)
    net.load_state_dict(synth.synth_state_dict(net.state_dict(), seed=6, style="default"), strict=True)
    net = net.to(DEV).eval().set_mode("h16")
    x = (torch.randint(0, 256, (1, 6, 1024, 1024), generator=torch.Generator().manual_seed(7)).float() / 127 - 1).to(DEV)
    with torch.no_grad():
        y = net(x).double().cpu()[:, :, ::8, ::8]
    yt = eager_tf32(net, x[:, :3].contiguous(), x[:, 3:].contiguous())[:, :, ::8, ::8]
    ref = torch.from_numpy(g["logits_f64ref_sub8"]).double()
    reduced_precision_bar(y, ref, "default", "xBD 1024 golden", yt)


def test_h16_graph_determinism_and_mode_isolation(levir_template):
    sd = synth.synth_state_dict(levir_template, seed=3, style="default")
    net = make_net(sd).set_mode("h16")
    a, b = (t.to(DEV) for t in synth.synth_pair(3, 256, 256, seed=40, kind="uniform"))
    with torch.no_grad():
        e1 = net(a, b).clone()
        assert torch.equal(net(a, b), e1)                     # two eager runs: bit-identical
        sa, sb = a.clone(), b.clone()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            net(sa, sb)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = net(sa, sb)
        sa.copy_(a); sb.copy_(b)
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, e1)                           # graph replay == eager
        net.set_mode("tf32x3")
        y_switched = net(a, b).clone()
        fresh = make_net(sd).set_mode("tf32x3")
        assert torch.equal(y_switched, fresh(a, b))           # h16 leaves nothing behind that a later mode reads


def test_c_host_runs_h16(tmp_path, levir_template):
    """examples/dahitra_infer.c with --flags DH_FLAGS_H16: logits bit-identical to the module's h16 forward"""
    from dahitra_b200 import _lib, checkpoints as CK
    from dahitra_b200.engine import MODES
    exe = _lib.build_example()
    sd = synth.synth_state_dict(levir_template, seed=3, style="default")
    x1, x2 = synth.synth_pair(2, 256, 256, seed=5, kind="uniform")
    wpath, ipath, opath = (str(tmp_path / n) for n in ("w.bin", "x.bin", "y.bin"))
    CK.export_state_dict_bin(sd, wpath)
    CK.write_pairs_bin(ipath, x1, x2)
    r = subprocess.run([exe, "--weights", wpath, "--input", ipath, "--output", opath, "--flags", str(MODES["h16"])],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout.strip())
    assert r.returncode == 0, r.stderr
    logits, cmap = CK.read_result_bin(opath)
    assert torch.equal(cmap.long(), logits.argmax(1))
    net = make_net(sd).set_mode("h16")
    with torch.no_grad():
        y = net(x1.to(DEV), x2.to(DEV)).cpu()
    assert torch.equal(y, logits)
