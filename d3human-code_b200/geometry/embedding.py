"""`Embedding`: drop-in for the reference module of the same name (geometry/embedding.py:4-38): x -> (x, sin(2^k x),
cos(2^k x), ...), k < N_freqs.  The arithmetic runs in libd3h_tets.so (d3h_mlp_embed); CUDA tensors only.  Twice
differentiable with respect to the points: under create_graph=True the backward pass is itself a Function whose gradient
runs in d3h_mlp_embed_second_backward / d3h_mlp_embed_tangent (a third derivative raises NotImplementedError)."""
from __future__ import annotations

import torch
from torch import nn

from .. import _cabi


class _EmbedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, n_freq):
        m = x.shape[0]
        c = 3 * (2 * n_freq + 1)
        out = torch.empty((m, c), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _cabi.check(_cabi.lib().d3h_mlp_embed(x.data_ptr(), m, n_freq, out.data_ptr(), c, c,
                                                  torch.cuda.current_stream(x.device).cuda_stream), "d3h_mlp_embed")
        ctx.save_for_backward(x)
        ctx.n_freq = n_freq
        return out

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        if torch.is_grad_enabled():          # create_graph=True: the adjoint as a differentiable Function of (x, g)
            return _EmbedGradFn.apply(x, g, ctx.n_freq), None
        return _embed_backward(x, g.contiguous().float(), ctx.n_freq), None


def _embed_backward(x, g, n_freq):
    gx = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _cabi.check(_cabi.lib().d3h_mlp_embed_backward(x.data_ptr(), x.shape[0], n_freq, g.data_ptr(), g.shape[1],
                                                       gx.data_ptr(), 0, torch.cuda.current_stream(x.device).cuda_stream),
                    "d3h_mlp_embed_backward")
    return gx


class _EmbedGradFn(torch.autograd.Function):
    """gx = E'(x)^T g, differentiable once: d/dx sum(v gx) = E''(x)[v]^T g (d3h_mlp_embed_second_backward), d/dg = E'(x) v
    (d3h_mlp_embed_tangent).  A third derivative raises NotImplementedError."""

    @staticmethod
    def forward(ctx, x, g, n_freq):
        g = g.contiguous().float()
        ctx.save_for_backward(x, g)
        ctx.n_freq = n_freq
        ctx.set_materialize_grads(False)
        return _embed_backward(x, g, n_freq)

    @staticmethod
    def backward(ctx, v):
        if torch.is_grad_enabled():
            raise NotImplementedError("d3human-code_b200 Embedding: no third derivative (create_graph=True through the second one)")
        if v is None:
            return None, None, None
        x, g = ctx.saved_tensors
        v = v.contiguous().float()
        m, c = x.shape[0], g.shape[1]
        L = _cabi.lib()
        with torch.cuda.device(x.device):
            st = torch.cuda.current_stream(x.device).cuda_stream
            hx = torch.empty_like(x)
            _cabi.check(L.d3h_mlp_embed_second_backward(x.data_ptr(), v.data_ptr(), m, ctx.n_freq, None, 0, g.data_ptr(), c,
                                                        hx.data_ptr(), st), "d3h_mlp_embed_second_backward")
            hg = None
            if ctx.needs_input_grad[1]:
                hg = torch.empty((m, c), dtype=torch.float32, device=x.device)
                _cabi.check(L.d3h_mlp_embed_tangent(x.data_ptr(), v.data_ptr(), m, ctx.n_freq, hg.data_ptr(), c, c, st),
                            "d3h_mlp_embed_tangent")
        return hx, hg, None


class Embedding(nn.Module):
    def __init__(self, in_channels, N_freqs, logscale=True):
        super().__init__()
        self.N_freqs = N_freqs
        self.in_channels = in_channels
        self.funcs = [torch.sin, torch.cos]
        self.out_channels = in_channels * (len(self.funcs) * N_freqs + 1)
        if logscale:
            self.freq_bands = 2 ** torch.linspace(0, N_freqs - 1, N_freqs)
        else:
            self.freq_bands = torch.linspace(1, 2 ** (N_freqs - 1), N_freqs)
        self.logscale = logscale

    def forward(self, x):
        if self.in_channels != 3 or not self.logscale:
            raise NotImplementedError("d3human-code_b200 Embedding: 3 input channels and logscale=True (what D3-Human uses)")
        if not x.is_cuda:
            raise RuntimeError("d3human-code_b200 has no CPU path: Embedding needs a CUDA tensor")
        shape = x.shape
        y = _EmbedFn.apply(x.reshape(-1, 3).contiguous().float(), self.N_freqs)
        return y.reshape(*shape[:-1], self.out_channels)
