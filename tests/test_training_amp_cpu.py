"""CPU: the mixed-precision surface of the training step — the 16-bit activation entry points of the C ABI (host-side checks
only) and GraphedTrainStep(amp=...) in its eager flat-buffer form against torch.amp.GradScaler."""
import copy
import ctypes
import os
import re

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EX = ("dahitra_pixel_decoder_train_fwd_ex", "dahitra_pixel_decoder_train_bwd_ex", "dahitra_tokenizer_train_fwd_ex",
      "dahitra_tokenizer_train_bwd_ex")


@pytest.fixture(scope="module")
def lib():
    from dahitra_b200 import _lib
    if _lib.needs_build():
        _lib.build()
    return _lib.load()


def test_act_dtype_entry_points_are_declared_and_bound():
    from dahitra_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "dahitra_b200.h")).read()
    for name in EX:
        assert re.search(rf"\b{name}\s*\(", hdr), name
        assert name in _lib.SIGNATURES, name
        assert _lib.SIGNATURES[name][1][-2] is ctypes.c_int, name          # act_dtype, just before the stream
    for macro, v in (("DH_ACT_F32", 0), ("DH_ACT_F16", 1), ("DH_ACT_BF16", 2)):
        assert re.search(rf"#define {macro}\s+{v}\b", hdr), macro
    from dahitra_b200 import training as T
    assert T._ACT == {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}


def test_unknown_act_dtype_is_refused_before_any_cuda_call(lib):
    buf = ctypes.create_string_buffer(1 << 12)
    p = ctypes.addressof(buf) + (-ctypes.addressof(buf) % 16)                   # a valid-looking 16-byte aligned pointer
    for bad in (3, -1, 7):
        assert lib.dahitra_pixel_decoder_train_fwd_ex(p, p, p, p, 2, 256, 4, 2, 0, bad, None) == -5
        assert lib.dahitra_pixel_decoder_train_bwd_ex(p, p, p, p, p, 2, 256, 4, 2, 1, bad, None) == -5
        assert lib.dahitra_tokenizer_train_fwd_ex(p, p, p, p, p, 2, 256, 0, bad, None) == -5
        assert lib.dahitra_tokenizer_train_bwd_ex(p, p, p, p, p, p, p, 2, 256, 1, bad, None) == -5
    # a known dtype goes on to the other checks: a pixel-major 16-bit tensor must be 16-byte aligned, a planar one 2-byte
    assert lib.dahitra_pixel_decoder_train_fwd_ex(p + 2, p, p, p, 2, 256, 4, 2, 1, 1, None) == -3
    assert lib.dahitra_tokenizer_train_fwd_ex(p + 1, p, p, p, p, 2, 256, 0, 2, None) == -3
    assert lib.dahitra_tokenizer_train_bwd_ex(p, p, p, p, p, p + 8, p, 2, 256, 1, 1, None) == -3


class _Net(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.a = torch.nn.Conv2d(3, 16, 3, padding=1)
        self.bn = torch.nn.BatchNorm2d(16)
        self.b = torch.nn.Conv2d(16, 2, 1)
        self.unused = torch.nn.Linear(4, 4)

    def forward(self, x):
        return self.b(F.relu(self.bn(self.a(x))))


def test_fp16_step_matches_gradscaler_loop_on_cpu():
    """the eager flat-buffer form of the fp16 step against the plain loop of torch.amp.GradScaler("cpu") with the same fused AdamW:
    started at scale 2^24 the first steps overflow and are skipped, and both loops see the same scale sequence and end with the
    same weights; the scaler state moves between the two in GradScaler.state_dict() form"""
    from dahitra_b200.train_graph import GraphedTrainStep
    torch.manual_seed(4)
    net = _Net()
    ref = copy.deepcopy(net).train()
    mk = lambda: (torch.randn(4, 3, 8, 8) * 4, torch.randint(0, 2, (4, 8, 8)))            # noqa: E731
    batches = [mk() for _ in range(7)]
    mk_opt = lambda ps: torch.optim.AdamW(ps, lr=1e-2, weight_decay=0.01, fused=True)      # noqa: E731
    ts = GraphedTrainStep(net, F.cross_entropy, batches[0], mk_opt, use_graph=False, amp=torch.float16)
    assert ts.scaler_state_dict() == torch.amp.GradScaler("cpu").state_dict()
    scaler = torch.amp.GradScaler("cpu", init_scale=2.0 ** 24)
    ts.load_scaler_state_dict(scaler.state_dict())
    opt = mk_opt([p for n, p in ref.named_parameters() if not n.startswith("unused")])
    scales, ref_scales = [], []
    for b in batches[1:]:
        l1 = float(ts.step(*b))
        scales.append(float(ts.scale))
        opt.zero_grad(set_to_none=True)
        with torch.autocast("cpu", dtype=torch.float16):
            l2 = F.cross_entropy(ref(b[0]), b[1])
        scaler.scale(l2).backward()
        scaler.step(opt)
        scaler.update()
        ref_scales.append(scaler.get_scale())
        assert l1 == float(l2.detach())
    print(f"[amp cpu] scales {scales}")
    assert scales == ref_scales and scales[0] < 2.0 ** 24 and scales[-1] == scales[-2]     # overflowed first, then settled
    for (k, v), w in zip(net.state_dict().items(), ref.state_dict().values()):
        assert torch.equal(v, w), k
    assert ts.scaler_state_dict() == scaler.state_dict()
    with pytest.raises(ValueError, match="growth_factor"):
        ts.load_scaler_state_dict(dict(scaler.state_dict(), growth_factor=4.0))


def test_fp16_step_refuses_an_optimizer_that_cannot_skip_on_the_device():
    from dahitra_b200.train_graph import GraphedTrainStep
    torch.manual_seed(5)
    net = _Net()
    before = copy.deepcopy(net.state_dict())
    batch = (torch.randn(2, 3, 8, 8), torch.randint(0, 2, (2, 8, 8)))
    with pytest.raises(ValueError, match="fused=True"):
        GraphedTrainStep(net, F.cross_entropy, batch, lambda ps: torch.optim.AdamW(ps, lr=1e-3), use_graph=False,
                         amp=torch.float16)
    for k, v in net.state_dict().items():                      # the refused construction leaves the module as it found it
        assert torch.equal(v, before[k]), k
    assert all(p.requires_grad and p.grad is None for p in net.parameters())
    # bf16 needs no scaler: any optimizer
    ts = GraphedTrainStep(net, F.cross_entropy, batch, lambda ps: torch.optim.AdamW(ps, lr=1e-3), use_graph=False,
                          amp=torch.bfloat16)
    assert ts.scaler_state_dict() == {} and torch.isfinite(ts.step(*batch))
    with pytest.raises(ValueError, match="amp must be"):
        GraphedTrainStep(net, F.cross_entropy, batch, lambda ps: torch.optim.AdamW(ps), use_graph=False, amp=torch.float64)
