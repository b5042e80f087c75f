"""GPU: mixed-precision training on the native kernels — fp16 / bf16 activation I/O of the training kernels (csrc/train_act.cuh),
the training route under autocast against the stock route and fp64 (reference xBD_code/train_unettransformer.py:435,474-476
runs its loop under autocast with a GradScaler), and GraphedTrainStep(amp=...) / net.graphed_training against eager AMP loops."""
import copy

import pytest
import torch
import torch.nn.functional as F

import emulate as E
from dahitra_b200 import training as T
from dahitra_b200.networks import define_G
from test_gpu_training import Args, _same_weights, rel

pytestmark = pytest.mark.gpu
DEV = "cuda"
DTYPES = [torch.float16, torch.bfloat16]
UNIT = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8}          # unit roundoff of the storage format


def _dn(dt):
    return str(dt).split(".")[-1]


@pytest.mark.parametrize("dtype", DTYPES, ids=_dn)
@pytest.mark.parametrize("heads,depth,B,N", [(4, 4, 3, 256), (4, 1, 2, 1024), (8, 8, 2, 4096), (8, 2, 1, 300), (4, 2, 2, 77)])
def test_pixel_decoder_16bit_io_is_the_fp32_kernel_rounded(dtype, heads, depth, B, N):
    """16-bit x / dout in, 16-bit out / dx: bit for bit the fp32 kernel on the up-cast inputs with out and dx rounded to the
    format, table gradients bit-identical; both layouts; against fp64 autograd within the format's rounding"""
    g = torch.Generator().manual_seed(heads * 100 + N + 7)
    x = (torch.randn(B, 32, N, generator=g)).to(dtype)
    tab = torch.randn(B, depth, T.train_tab_floats(heads), generator=g) * 0.15
    w = torch.randn(B, 32, N, generator=g).to(dtype)
    x16, t16 = x.to(DEV).requires_grad_(), tab.to(DEV).requires_grad_()
    y16 = T.pixel_decoder(x16, t16, heads)
    y16.backward(w.to(DEV))
    x32, t32 = x.float().to(DEV).requires_grad_(), tab.to(DEV).requires_grad_()
    y32 = T.pixel_decoder(x32, t32, heads)
    y32.backward(w.float().to(DEV))
    assert y16.dtype == dtype and x16.grad.dtype == dtype and t16.grad.dtype == torch.float32
    assert torch.equal(y16, y32.to(dtype)) and torch.equal(x16.grad, x32.grad.to(dtype)) and torch.equal(t16.grad, t32.grad)
    xd, td = x.double().requires_grad_(), tab.double().requires_grad_()
    yd = E.train_decoder_from_tables(xd, td, heads)
    (yd * w.double()).sum().backward()
    e = (rel(y16, yd), rel(x16.grad, xd.grad), rel(t16.grad, td.grad))
    print(f"[train decoder {_dn(dtype)}] heads {heads} depth {depth} B {B} N {N}: rel err out {e[0]:.2e} dx {e[1]:.2e} dtables {e[2]:.2e}")
    u = UNIT[dtype]
    assert e[0] <= u + 2e-6 and e[1] <= u + 1e-5 and e[2] < 1e-5, e
    h = 16 if N % 16 == 0 else 1
    if h > 1:                                                  # channels_last: 64 bytes per pixel, same bits
        xc = x.view(B, 32, h, N // h).to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_()
        tc = tab.to(DEV).requires_grad_()
        yc = T.pixel_decoder(xc, tc, heads)
        assert yc.dtype == dtype and yc.is_contiguous(memory_format=torch.channels_last) and torch.equal(yc.flatten(2), y16)
        yc.backward(w.to(DEV).view_as(yc).contiguous(memory_format=torch.channels_last))
        assert xc.grad.is_contiguous(memory_format=torch.channels_last)
        assert torch.equal(xc.grad.flatten(2), x16.grad) and torch.equal(tc.grad, t16.grad)


@pytest.mark.parametrize("dtype", DTYPES, ids=_dn)
@pytest.mark.parametrize("B,N", [(3, 256), (2, 1024), (2, 4096), (2, 300), (1, 77), (2, 16384)])
def test_semantic_tokens_16bit_io_is_the_fp32_kernel_rounded(dtype, B, N):
    """16-bit x in, fp32 tokens out, 16-bit dx: tokens and dW bit-identical to the fp32 kernel on the up-cast input, dx its fp32
    result rounded; both layouts; against fp64 autograd"""
    g = torch.Generator().manual_seed(N + 3)
    x = torch.randn(B, 32, N, generator=g).clamp_min(0).to(dtype)
    w = torch.randn(4, 32, 1, 1, generator=g) * 0.5
    dt = torch.randn(B, 4, 32, generator=g)
    x16, w16 = x.to(DEV).requires_grad_(), w.to(DEV).requires_grad_()
    tok16 = T.semantic_tokens(x16, w16)
    tok16.backward(dt.to(DEV))
    x32, w32 = x.float().to(DEV).requires_grad_(), w.to(DEV).requires_grad_()
    tok32 = T.semantic_tokens(x32, w32)
    tok32.backward(dt.to(DEV))
    assert tok16.dtype == torch.float32 and x16.grad.dtype == dtype
    assert torch.equal(tok16, tok32) and torch.equal(x16.grad, x32.grad.to(dtype)) and torch.equal(w16.grad, w32.grad)
    xd, wd = x.double().requires_grad_(), w.double().requires_grad_()
    a = torch.einsum("lc,bcn->bln", wd.view(4, 32), xd).softmax(-1)
    (torch.einsum("bln,bcn->blc", a, xd) * dt.double()).sum().backward()
    e = (rel(tok16, torch.einsum("bln,bcn->blc", a, xd)), rel(x16.grad, xd.grad), rel(w16.grad, wd.grad))
    print(f"[train tokens {_dn(dtype)}] B {B} N {N}: rel err tokens {e[0]:.2e} dx {e[1]:.2e} dW {e[2]:.2e}")
    assert e[0] < 2e-6 and e[1] <= UNIT[dtype] + 1e-5 and e[2] < 1e-5, e
    h = 16 if N % 16 == 0 else 1
    if h > 1:
        xc = x.view(B, 32, h, N // h).to(DEV).contiguous(memory_format=torch.channels_last).requires_grad_()
        wc = w.to(DEV).requires_grad_()
        tc = T.semantic_tokens(xc, wc)
        assert torch.equal(tc, tok16)
        tc.backward(dt.to(DEV))
        assert xc.grad.is_contiguous(memory_format=torch.channels_last)
        assert torch.equal(xc.grad.flatten(2), x16.grad) and torch.equal(wc.grad, w16.grad)


# ------------------------------------------------------------------------------------------------ the training step under autocast
LOSS_SCALE = 1024.0                           # exact power of two: keeps small fp16 gradients from flushing to zero, like GradScaler


def _amp_grads(net, xs, y, native, dtype):
    net.native_training = net.paired_trunk_training = native
    for p in net.parameters():
        p.grad = None
    if dtype == torch.float64:
        loss = F.cross_entropy(net(*xs), y)
        loss.backward()
    else:
        with torch.autocast("cuda", dtype=dtype):
            loss = F.cross_entropy(net(*xs), y)
        (loss * LOSS_SCALE).backward()
    s = 1.0 if dtype == torch.float64 else LOSS_SCALE
    return float(loss), {n: p.grad / s for n, p in net.named_parameters() if p.grad is not None}


def _amp_routes(net, xs, y, dtype, label):
    """loss and every parameter gradient of the native and the stock route under the same autocast, each against the network in
    fp64; the bar of test_gpu_training._compare_with_fp64: the native median error is at most 2x the stock median, and at most
    10 % of the tensors are more than 3x worse than stock"""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    sd0 = {k: v.clone() for k, v in net.state_dict().items()}
    ln, gn = _amp_grads(net, xs, y, True, dtype)
    net.load_state_dict(sd0)
    ls, gs = _amp_grads(net, xs, y, False, dtype)
    net.load_state_dict(sd0)
    net.double()
    l64, g64 = _amp_grads(net, [x.double() for x in xs], y, False, torch.float64)
    assert set(gn) == set(gs) == set(g64)
    errs = sorted(((rel(gn[k], g64[k]), rel(gs[k], g64[k]), k) for k in g64), reverse=True)
    en, es = sorted(e[0] for e in errs), sorted(e[1] for e in errs)
    med_n, med_s = en[len(en) // 2], es[len(es) // 2]
    out = [(k, a, b) for a, b, k in errs if a > 3 * b]
    dec = [(a, b) for a, b, k in errs if "transformer_decoder" in k or "conv_token" in k]
    print(f"[{label}] loss native {ln:.6f} stock {ls:.6f} fp64 {l64:.6f}")
    print(f"[{label}] {len(errs)} gradients vs fp64: native median {med_n:.2e} worst {en[-1]:.2e} ({errs[0][2]}); stock median "
          f"{med_s:.2e} worst {es[-1]:.2e}; {len(out)} tensors > 3x stock; decoder / tokenizer parameters ({len(dec)}): native worst "
          f"{max(d[0] for d in dec):.2e}, stock worst {max(d[1] for d in dec):.2e}")
    for k, a, b in out[:5]:
        print(f"[{label}]   > 3x stock: {k}: native {a:.2e} stock {b:.2e}")
    assert abs(ln - l64) <= 2e-2 * abs(l64) and abs(ls - l64) <= 2e-2 * abs(l64)
    assert med_n <= 2 * med_s, (med_n, med_s)
    assert len(out) <= 0.10 * len(errs), out[:8]


@pytest.mark.parametrize("dtype", DTYPES, ids=_dn)
def test_training_step_under_autocast_native_vs_stock(dtype):
    """LEVIR: under autocast the squeeze hands the tokenizer a 16-bit tensor while `x + pos` hands the decoders fp32"""
    torch.manual_seed(0)
    net = define_G(Args(), gpu_ids=[0]).train()
    g = torch.Generator(device=DEV).manual_seed(7)
    x1 = torch.rand(2, 3, 256, 256, device=DEV, generator=g) * 2 - 1
    x2 = torch.rand(2, 3, 256, 256, device=DEV, generator=g) * 2 - 1
    y = (torch.rand(2, 256, 256, device=DEV, generator=g) < 0.2).long()
    _amp_routes(net, [x1, x2], y, dtype, f"autocast {_dn(dtype)} LEVIR")


@pytest.mark.parametrize("dtype", DTYPES, ids=_dn)
def test_training_step_xbd_under_autocast_native_vs_stock(dtype):
    """xBD: the decoders see conv_decode's 16-bit output directly (no positional term at levels 4 and 3)"""
    from dahitra_b200 import xbd
    torch.manual_seed(1)
    net = xbd.BASE_Transformer_UNet(3, 5, with_pos='learned').to(DEV).train()
    g = torch.Generator(device=DEV).manual_seed(8)
    x = torch.rand(2, 6, 128, 160, device=DEV, generator=g) * 2 - 1
    y = torch.randint(0, 5, (2, 128, 160), device=DEV, generator=g)
    _amp_routes(net, [x], y, dtype, f"autocast {_dn(dtype)} xBD")


def test_reference_amp_loop_as_written_on_the_xbd_module():
    """the loop body of reference xBD_code/train_unettransformer.py:435,474-476 (autocast, scaler.scale(loss).backward(),
    scaler.step, scaler.update) runs on the native training route"""
    from dahitra_b200 import xbd
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = True, False
    torch.manual_seed(2)
    net = xbd.BASE_Transformer_UNet(3, 5, with_pos='learned').to(DEV).train()
    assert net.native_training
    w0 = {n: p.detach().clone() for n, p in net.named_parameters()}
    opt = torch.optim.AdamW(net.parameters(), lr=1e-4, weight_decay=1e-4)
    scaler = torch.amp.GradScaler("cuda")
    g = torch.Generator(device=DEV).manual_seed(9)
    for _ in range(3):
        x = torch.rand(2, 6, 128, 160, device=DEV, generator=g) * 2 - 1
        y = torch.randint(0, 5, (2, 128, 160), device=DEV, generator=g)
        opt.zero_grad()
        with torch.autocast("cuda"):
            out = net(x)
            loss = F.cross_entropy(out, y)
        assert out.dtype == torch.float16
        scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
    torch.cuda.synchronize()
    print(f"[reference AMP loop] loss {float(loss):.4f} scale {scaler.get_scale()}")
    moved = [n for n, p in net.named_parameters() if not torch.equal(p, w0[n])]
    assert all(torch.isfinite(p).all() for p in net.parameters())
    assert "transformer_decoder_3.layers.0.1.fn.fn.net.0.weight" in moved and "conv_token_3.weight" in moved
    assert len(moved) >= 0.5 * len(w0)


def _batches(g, n, b=2):
    return [(torch.rand(b, 3, 256, 256, device=DEV, generator=g) * 2 - 1, torch.rand(b, 3, 256, 256, device=DEV, generator=g) * 2 - 1,
             (torch.rand(b, 256, 256, device=DEV, generator=g) < 0.2).long()) for _ in range(n)]


@pytest.mark.parametrize("dtype", DTYPES, ids=_dn)
def test_graphed_amp_step_matches_the_eager_amp_loop(dtype):
    """GraphedTrainStep(amp=...) with fused AdamW against the eager autocast loop on a deep copy (fp16: with torch.amp.GradScaler,
    both started at scale 2^24, so the first steps overflow and are skipped): the same scale sequence, the same weights and
    BatchNorm statistics"""
    from dahitra_b200.train_graph import GraphedTrainStep
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = True, False
    torch.manual_seed(0)
    net = define_G(Args(), gpu_ids=[0]).train()
    ref = copy.deepcopy(net).train()
    batches = _batches(torch.Generator(device=DEV).manual_seed(13), 6)
    ts = GraphedTrainStep(net, F.cross_entropy, batches[0],
                          lambda ps: torch.optim.AdamW(ps, lr=1e-4, weight_decay=0.01, fused=True, capturable=True), amp=dtype)
    assert ts.use_graph
    fp16 = dtype == torch.float16
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 24, enabled=fp16)
    ts.load_scaler_state_dict(scaler.state_dict())
    opt = torch.optim.AdamW([p for p in ref.parameters() if p.requires_grad], lr=1e-4, weight_decay=0.01, fused=True)
    scales, ref_scales = [], []
    for b in batches[1:]:
        l1 = float(ts.step(*b))
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=dtype):
            l2 = F.cross_entropy(ref(b[0], b[1]), b[2])
        scaler.scale(l2).backward()
        scaler.step(opt)
        scaler.update()
        if fp16:
            scales.append(float(ts.scale))
            ref_scales.append(scaler.get_scale())
        assert abs(l1 - float(l2)) <= 1e-3 * abs(float(l2)), (l1, float(l2))
    torch.cuda.synchronize()
    print(f"[graphed amp step {_dn(dtype)}] scales {scales} eager {ref_scales}")
    assert scales == ref_scales
    if fp16:
        assert scales[0] < 2.0 ** 24 and ts.scaler_state_dict() == scaler.state_dict()
    _same_weights(net, ref, f"graphed amp step {_dn(dtype)}")


def test_graphed_route_under_autocast():
    """net.graphed_training inside the trainer's own AMP loop matches the plain route; a capture made under autocast is never
    replayed without it (nor the other way round): switching autocast runs the eager route"""
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = True, False
    torch.manual_seed(0)
    net = define_G(Args(), gpu_ids=[0]).train()
    ref = copy.deepcopy(net).train()
    net.graphed_training = True
    opts = [torch.optim.SGD(m.parameters(), lr=0.05, momentum=0.9, weight_decay=0.01) for m in (net, ref)]
    scalers = [torch.amp.GradScaler("cuda") for _ in (net, ref)]
    batches = _batches(torch.Generator(device=DEV).manual_seed(14), 5)
    for amp, b in zip((True, True, False, True, False), batches):
        losses = []
        for m, opt, sc in zip((net, ref), opts, scalers):
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.float16, enabled=amp):
                out = m(b[0], b[1])
                loss = F.cross_entropy(out, b[2])
            assert out.dtype == (torch.float16 if amp else torch.float32)
            sc.scale(loss).backward()
            sc.step(opt)
            sc.update()
            losses.append(float(loss))
        assert abs(losses[0] - losses[1]) <= 1e-3 * abs(losses[1]), (amp, losses)
    route = net.__dict__.get("_graphed_route")
    assert route is not None and route.key[-1] == (True, torch.float16)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        assert not route.matches(net, batches[0][:2])
    assert not route.matches(net, batches[0][:2])
    _same_weights(net, ref, "graphed route under autocast")
