"""Drop-in ``newUNetTrans`` network (LEVIR variant) and ``define_G`` factory.

Mirrors the reference interface for this path — same class name, constructor
arguments, state_dict keys (425) and ``forward(x1, x2) -> logits`` contract:

  * ``BASE_Transformer_UNet``   reference models/networks.py:1142-1357
  * ``define_G`` / ``init_net`` / ``init_weights``   reference models/networks.py:77-168

Inference (``eval()`` under ``torch.no_grad()``) runs on hand-written sm_100a
kernels through the C-ABI library (``include/dahitra_b200.h``).  There is no
CPU path and no PyTorch fallback for inference: a missing library or a CPU
tensor raises.  The training step (``train()`` / grad enabled) is autograd over the
same parameters: pixel decoders and tokenizer on native forward + backward kernels
(``dahitra_b200.training``), convolutions / BatchNorm on stock PyTorch (DESIGN.md,
"Training step").
"""
from __future__ import annotations

import functools
import os

import torch
from torch import nn
from torch.nn import init
import torch.nn.functional as F

from . import modules as M
from . import training as T
from .engine import NativeEngine

__all__ = ["BASE_Transformer_UNet", "define_G", "init_net", "init_weights"]

DIM = 32


class BASE_Transformer_UNet(nn.Module):
    """Siamese ResNet-18 trunk + per-scale tokenizer / token encoder / pixel decoder +
    UNet head.  Constructor signature of reference models/networks.py:1146-1154.

    Like the reference, the per-level depths/heads are fixed (decoder depth 4/4/8/1,
    heads 4/4/8/1) and ``dec_depth`` is stored but not used (networks.py:1221-1236).
    """

    VARIANT = "levir"

    def __init__(self, input_nc, output_nc, with_pos, resnet_stages_num=5,
                 token_len=4, token_trans=True, enc_depth=1, dec_depth=1,
                 dim_head=64, decoder_dim_head=64, tokenizer=True, if_upsample_2x=True,
                 pool_mode='max', pool_size=2, backbone='resnet18',
                 decoder_softmax=True, with_decoder_pos=None, with_decoder=True):
        super().__init__()
        if backbone != 'resnet18':
            raise NotImplementedError("dahitra_b200 builds the resnet18 trunk only (define_G's newUNetTrans)")
        if resnet_stages_num not in (3, 4, 5):
            raise NotImplementedError
        if input_nc != 3 or token_len != 4 or not tokenizer or not token_trans or not with_decoder \
                or enc_depth != 1 or dim_head != 64 or decoder_dim_head != 64 or not decoder_softmax:
            raise NotImplementedError(
                "dahitra_b200 implements the newUNetTrans configuration: input_nc=3, token_len=4, "
                "tokenizer/token_trans/with_decoder on, enc_depth=1, dim_head=decoder_dim_head=64, softmax decoder")
        # ---- ResNet_UNet part (reference networks.py:1086-1116) -------------------------------
        self.resnet = M.Trunk()
        self.resnet.load_imagenet_weights()        # resnet18(pretrained=True) of the reference, from a local file only (no download)
        self.relu = nn.ReLU()
        self.upsamplex2 = nn.Upsample(scale_factor=2)
        self.upsamplex4 = nn.Upsample(scale_factor=4, mode='bilinear')
        self.resnet_stages_num = resnet_stages_num
        self.if_upsample_2x = if_upsample_2x
        self.conv_pred = nn.Conv2d(384, 32, kernel_size=3, padding=1)       # dead weight, kept for checkpoints
        # ---- transformer part (reference networks.py:1160-1249); creation ORDER is part of the contract
        self.token_len, self.tokenizer, self.token_trans = token_len, tokenizer, token_trans
        self.with_decoder, self.with_pos = with_decoder, with_pos
        for k, cin in ((5, 256), (4, 128), (3, 64), (2, 64)):
            setattr(self, f"conv_squeeze_{k}", nn.Sequential(nn.Conv2d(cin, DIM, 1, bias=False), nn.ReLU()))
        for k in (5, 4, 3, 2):
            setattr(self, f"conv_token_{k}", nn.Conv2d(DIM, token_len, 1, bias=False))
        for k in (5, 4, 3, 2):
            setattr(self, f"conv_decode_{k}", nn.Conv2d(2 * DIM, DIM, 3, padding=1, bias=False))
        if with_pos == 'learned':
            for k in (5, 4, 3, 2):
                setattr(self, f"pos_embedding_{k}", nn.Parameter(torch.randn(1, token_len * 2, DIM)))
        self.with_decoder_pos = with_decoder_pos
        if with_decoder_pos == 'learned':
            for k, s in ((5, 16), (4, 32), (3, 64), (2, 64)):
                setattr(self, f"pos_embedding_decoder_{k}", nn.Parameter(torch.randn(1, DIM, s, s)))
        self.enc_depth, self.dec_depth = enc_depth, dec_depth
        self.dim_head, self.decoder_dim_head = dim_head, decoder_dim_head
        for k, heads, depth, dh in ((5, 4, 4, 64), (4, 4, 4, 64), (3, 8, 8, 64), (2, 1, 1, 32)):
            setattr(self, f"transformer_{k}", M.TokenEncoder(DIM, enc_depth, heads, dh, DIM))
            setattr(self, f"transformer_decoder_{k}", M.PixelDecoder(DIM, depth, heads, dh, DIM))
        self.conv_layer2_0 = M.two_layer_head(128, 32)
        self.conv_layer2 = nn.Sequential(nn.Conv2d(32, 32, 3, padding=1), nn.ReLU())
        self.conv_layer3 = nn.Sequential(nn.Conv2d(32, 32, 3, padding=1), nn.ReLU())
        self.conv_layer4 = nn.Sequential(nn.Conv2d(32, 32, 3, padding=1), nn.ReLU())
        self.classifier = nn.Conv2d(32, output_nc, 3, padding=1)
        self.output_nc = output_nc
        # training route: evaluate the pixel decoders in the collapsed algebra (modules.PixelDecoder.forward_collapsed: the same
        # function, ~16x smaller intermediates); False = the reference's as-written projections
        self.collapsed_training = True
        # training route: run the pixel decoders (forward AND backward) on the native sm_100a kernels whenever autograd is
        # recording (dahitra_b200/training.py, csrc/train_decoder.cu); False = stock torch ops as selected above
        self.native_training = True
        # training route: activations and 4-D parameters in torch.channels_last memory format (cuDNN's native layout on this GPU:
        # no NCHW <-> NHWC transposes around every convolution; the native decoder kernels read it pixel-major).  Shapes, values
        # and state_dict keys are unchanged — only strides
        self.channels_last_training = True
        # training route: both image sets through each trunk convolution as one batch, BatchNorm per set (_trunk_pair_autograd)
        self.paired_trunk_training = True
        # training route: replay forward and backward from CUDA graphs inside the caller's eager loop (training.GraphedRoute;
        # opt-in: the logits then live in a static buffer that the next training forward overwrites)
        self.graphed_training = False
        # native engine (lazy: weights are folded / re-laid-out on the first inference call)
        self._engine = NativeEngine()

    # ------------------------------------------------------------------ cache invalidation
    def invalidate_native_cache(self):
        """Drop the prepared (folded / re-laid-out) weights; they are rebuilt on the next inference call.
        Called automatically by train()/eval(), .to()/.cuda() and load_state_dict(); call it yourself after
        editing parameters in place any other way."""
        eng = self.__dict__.get("_engine")
        if eng is not None:
            eng.invalidate()

    def train(self, mode: bool = True):
        self.invalidate_native_cache()
        return super().train(mode)

    def _apply(self, fn, *a, **kw):
        self.invalidate_native_cache()
        self.__dict__.pop("_graphed_route", None)            # .to() / .double() replace the tensors the graphs captured
        return super()._apply(fn, *a, **kw)

    def __getstate__(self):
        st = dict(self.__dict__)
        st.pop("_graphed_route", None)                       # CUDA graphs are neither picklable nor copyable
        return st

    def __deepcopy__(self, memo):
        import copy
        cls = self.__class__
        new = cls.__new__(cls)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            if k != "_graphed_route":
                new.__dict__[k] = copy.deepcopy(v, memo)
        return new

    def load_state_dict(self, *a, **kw):
        self.invalidate_native_cache()
        return super().load_state_dict(*a, **kw)

    def set_mode(self, mode):
        """Precision mode of the native inference path: 'tf32x3' (default: tensor cores, error-compensated,
        fp32-grade), 'tf32' (what eager PyTorch does on this GPU by default), 'fp32' (strict, CUDA cores) — see
        dahitra_b200.engine.MODES.  Also settable per process with DAHITRA_MODE."""
        self._engine.set_mode(mode)
        return self

    def pos_shapes(self, H, W):
        """positions each decoder positional-embedding slot must cover for an HxW input"""
        if self.with_decoder_pos != 'learned':
            return {}
        return {f"DH_W_LV{k}_POS": (H // d) * (W // d) for k, d in ((5, 16), (4, 8), (3, 4))}

    # ------------------------------------------------------------------ checkpoint ballast
    _UNUSED_PREFIXES = ("conv_squeeze_2.", "conv_token_2.", "conv_decode_2.", "pos_embedding_2", "pos_embedding_decoder_2",
                        "transformer_2.", "transformer_decoder_2.", "conv_pred.", "resnet.layer4.", "resnet.fc.")

    def unused_parameter_names(self):
        """Parameters no forward ever reads — the reference module carries the same ballast (scale-2 tokenizer / transformer
        that `_forward_trans_module` is never called with, `conv_pred`, `resnet.layer4` / `fc`; models/networks.py:1106,1176-1238,
        1326-1351).  They never receive a gradient, which is why stock DistributedDataParallel needs
        `find_unused_parameters=True` on this network."""
        return [n for n, _ in self.named_parameters() if n.startswith(self._UNUSED_PREFIXES)]

    def freeze_unused_parameters(self):
        """requires_grad_(False) on `unused_parameter_names()`: DDP then runs without its per-step unused-parameter search.  The
        optimizer step is unchanged (AdamW skips parameters without a gradient either way).  Returns the names."""
        names = set(self.unused_parameter_names())
        for n, p in self.named_parameters():
            if n in names:
                p.requires_grad_(False)
        return sorted(names)

    # ------------------------------------------------------------------ forward
    def forward(self, x1, x2):
        if not (x1.is_cuda and x2.is_cuda):
            raise RuntimeError("dahitra_b200: inputs must be CUDA tensors — this framework has no CPU path")
        if self.training or torch.is_grad_enabled():
            return self._forward_training(x1, x2)
        return self._engine.forward_pair(self, x1, x2)

    def _forward_training(self, *xs):
        """the autograd route, replayed from CUDA graphs when `graphed_training` is on (training.GraphedRoute)"""
        if self.training and torch.is_grad_enabled() and not torch.cuda.is_current_stream_capturing() \
                and (getattr(self, "graphed_training", False) or os.environ.get("DAHITRA_GRAPH_TRAINING") == "1"):
            route = self.__dict__.get("_graphed_route")
            if route is None:
                route = self.__dict__["_graphed_route"] = T.GraphedRoute(self, xs)
            if route.matches(self, xs):
                return route(*xs)
        return self._forward_autograd(*xs)

    # ------------------------------------------------------------------ training route (autograd; native decoder / tokenizer kernels)
    def _trunk_autograd(self, x):
        r = self.resnet
        x2 = F.relu(r.bn1(r.conv1(x)))
        x4 = r.layer1(r.maxpool(x2))
        x8 = r.layer2(x4)
        x16 = r.layer3(r.maxpool(x8))
        return x2, x4, x8, x16

    def _level_autograd(self, f1, f2, k, f12=None):
        """f12: optional batch [f1 | f2] already in one tensor (paired trunk)"""
        sq, tk = getattr(self, f"conv_squeeze_{k}"), getattr(self, f"conv_token_{k}")
        enc, dec = getattr(self, f"transformer_{k}"), getattr(self, f"transformer_decoder_{k}")

        def tokens(x):
            a = tk(x).flatten(2).softmax(-1)
            return a @ x.flatten(2).transpose(1, 2)

        native = getattr(self, "native_training", True) and torch.is_grad_enabled()
        pos = getattr(self, f"pos_embedding_decoder_{k}") if self.with_decoder_pos == 'learned' else None

        def decode(x, m):
            b, c, h, w = x.shape
            if pos is not None:
                x = x + pos
            run = dec.forward_collapsed if getattr(self, "collapsed_training", True) else dec
            return run(x.flatten(2).transpose(1, 2), m).transpose(1, 2).reshape(b, c, h, w)

        def decode_native(x, tab):                           # NCHW / channels_last are the kernels' two layouts: no transposes
            if pos is not None:
                x = x + pos
            return T.pixel_decoder(x, tab, dec.heads)

        conv_decode = getattr(self, f"conv_decode_{k}")
        if native:
            # both image sets as one batch (the squeeze has no BatchNorm): tokenizer, ONE table build for the level's three
            # decoder calls, one decoder launch for x1 | x2 and one for the difference features
            nb = f1.shape[0]
            x12 = sq(torch.cat([f1, f2]) if f12 is None else f12)
            t12 = T.semantic_tokens(x12, tk.weight)
            # tokens, token encoder and tables are a few KB: fp32 even under autocast (16 bits would only cost accuracy)
            with torch.autocast("cuda", enabled=False):
                tok = torch.cat([t12[:nb], t12[nb:]], dim=1)
                if self.with_pos:
                    tok = tok + getattr(self, f"pos_embedding_{k}")
                t1, t2 = enc(tok).chunk(2, dim=1)
                tab = dec.train_tables(torch.cat([t1, t2, (t2 - t1).abs()]))
            y12 = decode_native(x12, tab[:2 * nb])
            return decode_native(conv_decode(torch.cat([y12[:nb], y12[nb:]], dim=1)), tab[2 * nb:])
        x1, x2 = sq(f1), sq(f2)
        tok = torch.cat([tokens(x1), tokens(x2)], dim=1)
        if self.with_pos:
            tok = tok + getattr(self, f"pos_embedding_{k}")
        t1, t2 = enc(tok).chunk(2, dim=1)
        x1, x2 = decode(x1, t1), decode(x2, t2)
        return decode(conv_decode(torch.cat([x1, x2], dim=1)), (t2 - t1).abs())

    def _channels_last(self, *xs):
        if not getattr(self, "channels_last_training", True):
            return xs
        if not self.resnet.conv1.weight.is_contiguous(memory_format=torch.channels_last):
            for p in self.parameters():
                if p.dim() == 4:
                    p.data = p.data.contiguous(memory_format=torch.channels_last)
                    if p.grad is not None:
                        p.grad.data = p.grad.data.contiguous(memory_format=torch.channels_last)
        return tuple(x.contiguous(memory_format=torch.channels_last) for x in xs)

    def _trunk_pair_autograd(self, x12, nb):
        """Both image sets through every convolution as ONE batch (convolutions are per-sample), BatchNorm applied per set:
        batch statistics and the running-stat updates are exactly the reference's two forward_single passes (set 1, then
        set 2, per layer), with half the convolution launches and twice the rows per launch."""
        r = self.resnet

        def bn2(bn, y):
            return torch.cat([bn(y[:nb]), bn(y[nb:])])

        def stage(blocks, x):
            for blk in blocks:
                idt = x if blk.downsample is None else bn2(blk.downsample[1], blk.downsample[0](x))
                y = F.relu(bn2(blk.bn1, blk.conv1(x)))
                x = F.relu(bn2(blk.bn2, blk.conv2(y)) + idt)
            return x

        x2 = F.relu(bn2(r.bn1, r.conv1(x12)))
        x4 = stage(r.layer1, r.maxpool(x2))
        x8 = stage(r.layer2, x4)
        x16 = stage(r.layer3, r.maxpool(x8))
        return x2, x4, x8, x16

    def _forward_autograd(self, x1, x2):
        x1, x2 = self._channels_last(x1, x2)
        nb = x1.shape[0]
        if getattr(self, "paired_trunk_training", True) and torch.is_grad_enabled():
            t = self._trunk_pair_autograd(torch.cat([x1, x2]), nb)
            a, b = [f[:nb] for f in t], [f[nb:] for f in t]
        else:
            a, b = self._trunk_autograd(x1), self._trunk_autograd(x2)   # two passes: BN batch stats per image set
            t = (None,) * 4
        up = self.upsamplex2
        o5 = up(self._level_autograd(a[3], b[3], 5, f12=t[3]))
        o4 = self.conv_layer4(up(self._level_autograd(a[2], b[2], 4, f12=t[2]) + o5))
        o3 = self.conv_layer3(up(self._level_autograd(a[1], b[1], 3, f12=t[1]) + o4))
        o2 = self.conv_layer2(up(self.conv_layer2_0(torch.cat([a[0], b[0]], 1)) + o3))
        return self.classifier(o2)


# ----------------------------------------------------------------------------- factory
def init_weights(net, init_type='normal', init_gain=0.02):
    """Same contract as reference models/networks.py:77-108: every module whose class name
    contains 'Conv' or 'Linear' gets N(0, gain) weights / zero bias; BatchNorm2d gets N(1, gain)."""
    makers = {'normal': lambda w: init.normal_(w, 0.0, init_gain),
              'xavier': lambda w: init.xavier_normal_(w, gain=init_gain),
              'kaiming': lambda w: init.kaiming_normal_(w, a=0, mode='fan_in'),
              'orthogonal': lambda w: init.orthogonal_(w, gain=init_gain)}
    if init_type not in makers:
        raise NotImplementedError('initialization method [%s] is not implemented' % init_type)

    def visit(m):
        name = type(m).__name__
        if hasattr(m, 'weight') and ('Conv' in name or 'Linear' in name):
            makers[init_type](m.weight.data)
            if getattr(m, 'bias', None) is not None:
                init.constant_(m.bias.data, 0.0)
        elif 'BatchNorm2d' in name:
            init.normal_(m.weight.data, 1.0, init_gain)
            init.constant_(m.bias.data, 0.0)

    print('initialize network with %s' % init_type)
    net.apply(visit)
    if hasattr(net, "invalidate_native_cache"):
        net.invalidate_native_cache()


def init_net(net, init_type='normal', init_gain=0.02, gpu_ids=[]):
    """reference models/networks.py:111-127.  One process drives one GPU here: several gpu_ids are
    rejected instead of wrapping in nn.DataParallel (which cannot replicate the reference model
    either — its per-level module lists are plain Python lists; SURVEY.md §2.1)."""
    if len(gpu_ids) > 0:
        assert torch.cuda.is_available()
        if len(gpu_ids) > 1:
            raise NotImplementedError("dahitra_b200 runs one process per GPU (torchrun); pass a single gpu id")
        net.to(gpu_ids[0])
    init_weights(net, init_type, init_gain=init_gain)
    return net


def define_G(args, init_type='normal', init_gain=0.02, gpu_ids=[]):
    """reference models/networks.py:130-168, restricted to the in-scope ``newUNetTrans`` branch."""
    if args.net_G == 'newUNetTrans':
        net = BASE_Transformer_UNet(input_nc=3, output_nc=2, token_len=4, resnet_stages_num=4,
                                    with_pos='learned', with_decoder_pos='learned', enc_depth=1, dec_depth=8)
    else:
        raise NotImplementedError('Generator model name [%s] is not built by dahitra_b200 '
                                  '(only newUNetTrans is in scope)' % args.net_G)
    return init_net(net, init_type, init_gain, gpu_ids)
