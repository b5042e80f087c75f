"""Native pieces of the TRAINING step (SURVEY.md §8 f4): ``torch.autograd.Function``s over hand-written sm_100a kernels.

The training step of the reference (models/trainer.py:247-262: forward, CE loss, backward, optimizer step) runs on the drop-in
module's autograd route.  What that route spends its device time on is the pixel decoders
(``profiles/r02_train_step_ablation.json``: 27 of 36 ms of forward + backward at batch 8), so those run natively:

* ``semantic_tokens(x, w_tok)`` — the tokenizer (reference models/networks.py:1273-1280: 1x1 conv to 4 maps, softmax over the
  pixels, weighted sum to 4 tokens) as one partial + merge forward and ONE backward pass over x (csrc/train_tokens.cu).
* ``pixel_decoder(x, tables, heads)`` — all layers of one ``TransformerDecoder`` call (reference models/help_funcs.py:66-114,
  170-186) for every pixel in ONE forward launch, and the whole backward in ONE launch that returns dL/dx and the gradient of the
  per-(image, layer) tables (``modules.PixelDecoder.train_tables`` builds those from the parameters and the 4 memory tokens with
  differentiable torch ops on tensors of a few KB, so autograd carries the table gradients on to Wq / Wk / Wv / Wo, the
  LayerNorm affines, the MLP, the tokens and everything upstream of the tokens).

Mixed precision: both accept x in fp32, fp16 or bf16 (what autocast hands them) and keep x's dtype for the activations that
leave them (the decoder's output, every dL/dx); the kernels convert on load and store and compute in fp32.  Tables, tokens and
w_tok are fp32 (converted at the boundary, so their gradients flow back through the conversion).

There is no fallback: the functions raise if the CUDA library is missing or the tensors are not on a GPU.
"""
from __future__ import annotations

import contextlib

import torch

from . import _lib


def train_tab_floats(heads: int) -> int:
    """DH_TRAIN_TAB_FLOATS of include/dahitra_b200.h"""
    return 65 * 4 * heads + 96 + 2048


_ACT = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}         # DH_ACT_* of include/dahitra_b200.h


def _act(x):
    if x.dtype not in _ACT:
        raise RuntimeError(f"dahitra_b200.training: activations must be fp32, fp16 or bf16, got {x.dtype}")
    return _ACT[x.dtype]


def _layout(t):
    """(tensor in a layout the kernels read, pixel_major flag): (B, 32, N) / NCHW-contiguous -> planar; a 4-D tensor in
    torch.channels_last memory format -> pixel-major, without a copy; anything else is made NCHW-contiguous."""
    if t.dim() == 4 and not t.is_contiguous() and t.is_contiguous(memory_format=torch.channels_last):
        return t, 1
    return t.contiguous(), 0


class _PixelDecoderTrain(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, tables, heads):
        if not (x.is_cuda and tables.is_cuda):
            raise RuntimeError("dahitra_b200.training: tensors must be on a CUDA device — there is no CPU path")
        act = _act(x)
        if tables.dtype != torch.float32:
            raise RuntimeError("dahitra_b200.training: the decoder tables must be fp32")
        B, C = x.shape[:2]
        N = x[0, 0].numel()
        depth = tables.shape[1]
        if C != 32 or tables.shape[0] != B or tables.shape[2] != train_tab_floats(heads):
            raise RuntimeError(f"pixel_decoder: x {tuple(x.shape)} / tables {tuple(tables.shape)} do not fit heads={heads}")
        x, pm = _layout(x)
        tables = tables.contiguous()
        lib = _lib.load()
        xs = torch.empty((depth, B, 32, N), dtype=torch.float32, device=x.device)
        out = torch.empty_like(x)                           # same memory format as x
        with torch.cuda.device(x.device):
            rc = lib.dahitra_pixel_decoder_train_fwd_ex(x.data_ptr(), tables.data_ptr(), xs.data_ptr(), out.data_ptr(), B, N, heads,
                                                        depth, pm, act, torch.cuda.current_stream(x.device).cuda_stream)
        _lib.check(rc, "dahitra_pixel_decoder_train_fwd_ex")
        ctx.save_for_backward(xs, tables)
        ctx.heads, ctx.dtype = heads, x.dtype
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dout):
        xs, tables = ctx.saved_tensors
        depth, B, _, N = xs.shape
        lib = _lib.load()
        dout, pm = _layout(dout.to(ctx.dtype))
        nblk = lib.dahitra_pixel_decoder_train_blocks(N)
        dx = torch.empty_like(dout)
        partial = torch.empty((B, nblk, depth, tables.shape[2]), dtype=torch.float32, device=dout.device)
        with torch.cuda.device(dout.device):
            rc = lib.dahitra_pixel_decoder_train_bwd_ex(dout.data_ptr(), xs.data_ptr(), tables.data_ptr(), dx.data_ptr(),
                                                        partial.data_ptr(), B, N, ctx.heads, depth, pm, _ACT[ctx.dtype],
                                                        torch.cuda.current_stream(dout.device).cuda_stream)
        _lib.check(rc, "dahitra_pixel_decoder_train_bwd_ex")
        return dx, partial.sum(1), None


def pixel_decoder(x: torch.Tensor, tables: torch.Tensor, heads: int) -> torch.Tensor:
    """x: (B, 32, N) or (B, 32, h, w) fp32 / fp16 / bf16 CUDA — NCHW-contiguous (the kernels' channel-planar layout) or, 4-D
    only, in torch.channels_last memory format (read pixel-major, no copy); tables (B, depth, DH_TRAIN_TAB_FLOATS(heads)), used
    in fp32.  Returns a tensor of x's shape, dtype and memory format.  Differentiable in x and tables (first order)."""
    return _PixelDecoderTrain.apply(x, tables.float(), heads)


class _SemanticTokensTrain(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w_tok):
        if not (x.is_cuda and w_tok.is_cuda):
            raise RuntimeError("dahitra_b200.training: tensors must be on a CUDA device — there is no CPU path")
        act = _act(x)
        if w_tok.dtype != torch.float32:
            raise RuntimeError("dahitra_b200.training: w_tok must be fp32")
        B, C = x.shape[:2]
        N = x[0, 0].numel()
        if C != 32 or w_tok.numel() != 128:
            raise RuntimeError(f"semantic_tokens: x {tuple(x.shape)} / w_tok {tuple(w_tok.shape)}: 32 channels and 4 tokens expected")
        x, pm = _layout(x)
        w = w_tok.reshape(4, 32).contiguous()
        lib = _lib.load()
        part = torch.empty((B, lib.dahitra_tokenizer_train_chunks(N), 4, 34), dtype=torch.float32, device=x.device)
        tok = torch.empty((B, 4, 32), dtype=torch.float32, device=x.device)
        stats = torch.empty((B, 4, 2), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            rc = lib.dahitra_tokenizer_train_fwd_ex(x.data_ptr(), w.data_ptr(), part.data_ptr(), tok.data_ptr(), stats.data_ptr(), B, N,
                                                    pm, act, torch.cuda.current_stream(x.device).cuda_stream)
        _lib.check(rc, "dahitra_tokenizer_train_fwd_ex")
        ctx.save_for_backward(x, w, tok, stats)
        ctx.pm, ctx.w_shape, ctx.act = pm, w_tok.shape, act
        return tok

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dtok):
        x, w, tok, stats = ctx.saved_tensors
        B = x.shape[0]
        N = x[0, 0].numel()
        lib = _lib.load()
        dtok = dtok.float().contiguous()
        dx = torch.empty_like(x)
        dwp = torch.empty((B, lib.dahitra_tokenizer_train_chunks(N), 4, 32), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            rc = lib.dahitra_tokenizer_train_bwd_ex(x.data_ptr(), w.data_ptr(), tok.data_ptr(), stats.data_ptr(), dtok.data_ptr(),
                                                    dx.data_ptr(), dwp.data_ptr(), B, N, ctx.pm, ctx.act,
                                                    torch.cuda.current_stream(x.device).cuda_stream)
        _lib.check(rc, "dahitra_tokenizer_train_bwd_ex")
        return dx, dwp.sum((0, 1)).reshape(ctx.w_shape)


def semantic_tokens(x: torch.Tensor, w_tok: torch.Tensor) -> torch.Tensor:
    """x: (B, 32, N) or (B, 32, h, w) fp32 / fp16 / bf16 CUDA (NCHW-contiguous or channels_last), w_tok: conv_token_k.weight
    (4, 32, 1, 1), used in fp32 -> fp32 tokens (B, 4, 32).  Differentiable in both (first order); dL/dx has x's dtype."""
    return _SemanticTokensTrain.apply(x, w_tok.float())


# ------------------------------------------------------------------------------------------------ graphed autograd route
class _Route(torch.nn.Module):
    """the module's training forward as a callable torch.cuda.make_graphed_callables can wrap (it needs an nn.Module to find
    the parameters)"""

    def __init__(self, net):
        super().__init__()
        self.net = net

    def forward(self, *xs):
        return self.net._forward_autograd(*xs)


class GraphedRoute:
    """forward AND backward of the module's training route as two replayed CUDA graphs inside an ordinary eager training loop
    (torch.cuda.make_graphed_callables): the reference trainer (models/trainer.py:247-262) keeps computing its loss, calling
    backward() and stepping its optimizer eagerly, but the ~1200 launches of the network itself are issued by two graph
    replays.  Built on the first training forward of a given input shape when `net.graphed_training` is set (or
    DAHITRA_GRAPH_TRAINING=1); other shapes (e.g. a last, smaller batch) run the eager route.  The autocast state (on / off and
    its dtype) is part of what was captured: a capture made under autocast (captured with the autocast weight cache off, which
    graphs require) is replayed only under the same autocast, an fp32 capture only without it; the other state runs eagerly.  The returned logits live in the
    graph's static output buffer: they are overwritten by the next training forward, like any graphed callable's."""

    def __init__(self, net, xs):
        self.key = self._key(net, xs)
        if hasattr(net, "_channels_last"):
            net._channels_last()                                      # parameter layouts settle before anything is captured
        buffers = [(b, b.clone()) for b in net.buffers()]             # the warm-up / capture passes must leave no trace
        grads = [(p, p.grad) for p in net.parameters()]
        sample = tuple(x.detach().clone() for x in xs)
        amp = self.key[-1]
        with torch.autocast("cuda", dtype=amp[1], cache_enabled=False) if amp[0] else contextlib.nullcontext():
            self.call = torch.cuda.make_graphed_callables(_Route(net), sample, allow_unused_input=True)
        with torch.no_grad():
            for b, s in buffers:
                b.copy_(s)
        for p, g in grads:
            p.grad = g

    @staticmethod
    def _key(net, xs):
        # input signature + the route switches that were captured (changing one of them afterwards falls back to the eager route)
        flags = tuple(bool(getattr(net, f, True)) for f in ("native_training", "channels_last_training", "paired_trunk_training",
                                                            "collapsed_training"))
        amp = torch.is_autocast_enabled("cuda")
        return tuple((tuple(x.shape), x.dtype, x.device) for x in xs) + (flags, (amp, torch.get_autocast_dtype("cuda") if amp else None))

    def matches(self, net, xs):
        return self.key == self._key(net, xs) and not any(x.requires_grad for x in xs)

    def __call__(self, *xs):
        return self.call(*xs)
