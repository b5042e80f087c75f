"""xBD variant of the drop-in network (config 3: 1024x1024 pre/post pair, 5-class damage map).

Mirrors ``BASE_Transformer_UNet`` of reference xBD_code/zoo/model_transformer_encoding.py:242-449:
  * ``forward(x)`` with x = cat[pre, post] on channels (:409-412)
  * one pixel-decoder pass per level on ``conv_decode(cat[squeeze(x1), squeeze(x2)])`` (:385-406)
  * positional terms only on the H/16 level, taken from ``pos_embedding_3`` /
    ``pos_embedding_decoder_3`` (64x64 => H = W = 1024 when with_decoder_pos='learned') (:358-383)
  * per-level containers are ``nn.ModuleList``s, which adds alias keys to the state_dict
    (700 keys in total) — reproduced so xBD checkpoints load strictly.
"""
from __future__ import annotations

import contextlib

import torch
from torch import nn
import torch.nn.functional as F

from . import modules as M
from . import training as T
from .engine import NativeEngine
from .networks import BASE_Transformer_UNet as _LevirNet

DIM = 32


class BASE_Transformer_UNet(_LevirNet):
    VARIANT = "xbd"

    def __init__(self, input_nc, output_nc, with_pos=None, resnet_stages_num=5,
                 token_len=4, token_trans=True, enc_depth=1, dec_depth=1,
                 dim_head=64, decoder_dim_head=64, tokenizer=True, if_upsample_2x=True,
                 pool_mode='max', pool_size=2, backbone='resnet18',
                 decoder_softmax=True, with_decoder_pos=None, with_decoder=True):
        nn.Module.__init__(self)
        if backbone != 'resnet18' or input_nc != 3 or token_len != 4 or not tokenizer or not token_trans \
                or not with_decoder or enc_depth != 1 or dim_head != 64 or decoder_dim_head != 64 or not decoder_softmax:
            raise NotImplementedError("dahitra_b200.xbd implements the configuration of xBD_code/train.py:44-45 only")
        self.resnet = M.Trunk()
        self.resnet.load_imagenet_weights()        # resnet18(pretrained=True) of the reference, from a local file only (no download)
        self.relu = nn.ReLU()
        self.upsamplex2 = nn.Upsample(scale_factor=2)
        self.upsamplex4 = nn.Upsample(scale_factor=4, mode='bilinear')
        self.resnet_stages_num, self.if_upsample_2x = resnet_stages_num, if_upsample_2x
        self.conv_pred = nn.Conv2d(384, 32, kernel_size=3, padding=1)
        self.token_len, self.tokenizer, self.token_trans = token_len, tokenizer, token_trans
        self.with_decoder, self.with_pos = with_decoder, with_pos

        def group(prefix, make):
            mods = {k: make(k) for k in (5, 4, 3, 2)}
            for k in (5, 4, 3, 2):
                setattr(self, f"{prefix}_{k}", mods[k])
            return nn.ModuleList([mods[2], mods[3], mods[4], mods[5]])

        cin = {5: 256, 4: 128, 3: 64, 2: 64}
        self.conv_squeeze_layers = group("conv_squeeze", lambda k: nn.Sequential(
            nn.Conv2d(cin[k], DIM, 1, bias=False), nn.ReLU()))
        self.conv_tokens_layers = group("conv_token", lambda k: nn.Conv2d(DIM, token_len, 1, bias=False))
        self.conv_decode_layers = group("conv_decode", lambda k: nn.Conv2d(2 * DIM, DIM, 3, padding=1, bias=False))
        if with_pos == 'learned':
            for k in (5, 4, 3):
                setattr(self, f"pos_embedding_{k}", nn.Parameter(torch.randn(1, token_len * 2, DIM)))
        self.with_decoder_pos = with_decoder_pos
        if with_decoder_pos == 'learned':
            for k, s in ((5, 16), (4, 32), (3, 64)):
                setattr(self, f"pos_embedding_decoder_{k}", nn.Parameter(torch.randn(1, DIM, s, s)))
        self.enc_depth, self.dec_depth = enc_depth, dec_depth
        self.dim_head, self.decoder_dim_head = dim_head, decoder_dim_head
        enc, dec = {}, {}
        for k, heads, depth, dh in ((5, 4, 4, 64), (4, 4, 4, 64), (3, 8, 8, 64), (2, 1, 1, 32)):
            enc[k] = M.TokenEncoder(DIM, enc_depth, heads, dh, DIM)
            setattr(self, f"transformer_{k}", enc[k])
            dec[k] = M.PixelDecoder(DIM, depth, heads, dh, DIM)
            setattr(self, f"transformer_decoder_{k}", dec[k])
        self.transformer_layers = nn.ModuleList([enc[2], enc[3], enc[4], enc[5]])
        self.transformer_decoder_layers = nn.ModuleList([dec[2], dec[3], dec[4], dec[5]])
        self.conv_layer2_0 = M.two_layer_head(128, 32)
        self.conv_layer2 = nn.Sequential(nn.Conv2d(32, 32, 3, padding=1), nn.ReLU())
        self.conv_layer3 = nn.Sequential(nn.Conv2d(32, 32, 3, padding=1), nn.ReLU())
        self.conv_layer4 = nn.Sequential(nn.Conv2d(32, 32, 3, padding=1), nn.ReLU())
        self.classifier = nn.Conv2d(32, output_nc, 3, padding=1)
        self.output_nc = output_nc
        self.collapsed_training = True          # training route: pixel decoders in the collapsed algebra (see networks.py)
        self.native_training = True             # ... on the native kernels whenever autograd is recording (training.py)
        self.channels_last_training = True      # ... with activations / 4-D parameters in torch.channels_last (see networks.py)
        self.paired_trunk_training = True       # ... and both image sets through each trunk convolution as one batch
        self.graphed_training = False           # opt-in: forward / backward replayed from CUDA graphs (training.GraphedRoute)
        self._engine = NativeEngine()

    def pos_shapes(self, H, W):
        if self.with_decoder_pos != 'learned':
            return {}
        return {"DH_W_LV5_POS": (H // 16) * (W // 16)}

    def forward(self, x):
        if not x.is_cuda:
            raise RuntimeError("dahitra_b200: inputs must be CUDA tensors — this framework has no CPU path")
        if self.training or torch.is_grad_enabled():
            return self._forward_training(x[:, :3], x[:, 3:])
        return self._engine.forward_stacked(self, x)

    # training route: same chain as the LEVIR class except for the trans-module (one decoder pass)
    def _level_autograd(self, f1, f2, k, f12=None):
        sq, tk = getattr(self, f"conv_squeeze_{k}"), getattr(self, f"conv_token_{k}")
        enc, dec = getattr(self, f"transformer_{k}"), getattr(self, f"transformer_decoder_{k}")

        def tokens(x):
            return tk(x).flatten(2).softmax(-1) @ x.flatten(2).transpose(1, 2)

        native = getattr(self, "native_training", True) and torch.is_grad_enabled()
        if native:
            nb = f1.shape[0]
            x12 = sq(torch.cat([f1, f2]) if f12 is None else f12)
            t12 = T.semantic_tokens(x12, tk.weight)
            x1, x2 = x12[:nb], x12[nb:]
            tok = torch.cat([t12[:nb], t12[nb:]], dim=1)
        else:
            x1, x2 = sq(f1), sq(f2)
            tok = torch.cat([tokens(x1), tokens(x2)], dim=1)
        # native route: tokens, token encoder and tables are a few KB, fp32 even under autocast (see networks.py)
        with torch.autocast("cuda", enabled=False) if native else contextlib.nullcontext():
            if self.with_pos and k == 5:
                tok = tok + self.pos_embedding_3
            t1, t2 = enc(tok).chunk(2, dim=1)
            tab = dec.train_tables((t2 - t1).abs()) if native else None
        dx = getattr(self, f"conv_decode_{k}")(torch.cat([x1, x2], dim=1))
        if self.with_decoder_pos == 'learned' and k == 5:
            dx = dx + self.pos_embedding_decoder_3
        b, c, h, w = dx.shape
        if native:
            return T.pixel_decoder(dx, tab, dec.heads)
        run = dec.forward_collapsed if getattr(self, "collapsed_training", True) else dec
        return run(dx.flatten(2).transpose(1, 2), (t2 - t1).abs()).transpose(1, 2).reshape(b, c, h, w)
