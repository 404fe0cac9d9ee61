"""Fused GRU sequence head: last hidden state of an nn.GRU (one layer, or a stack) through libsldm_sage.so.

Reference: src/models/grusage.py:55-60 (the nn.GRU it builds) and :160-161 (`gru_out, hlast = self.gru(x);
x = hlast[-1]`).  The parameters stay in the caller's own `torch.nn.GRU` module (same state-dict keys
`gru.weight_ih_l0` ...), only the arithmetic moves: one kernel runs all T steps of a tile of sequences on one SM
(csrc/gru.cu), the backward is two more kernels (the reverse recurrence, then dW_hh as a persistent split-K product).  Shapes the kernels do not cover
(`fused_gru_eligible` is False) stay on torch's library GRU in the caller -- a GPU library layer, as in the reference.
A stacked module (num_layers > 1) goes through `gru_stack_last_hidden` (`fused_gru_stack_eligible`): the same kernels
layer by layer, each layer above the first fed by an input projection of the layer below's output sequence.
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

from ._lib import lib, check
from .ops import _ptr, _require_cuda, _stream


def fused_gru_eligible(gru: torch.nn.GRU, x: torch.Tensor) -> bool:
    """True when `gru(x)[1][-1]` can run on the fused kernels: one unidirectional batch-first layer with biases,
    fp32 CUDA input [N, T, I], hidden size 32 / 64 / 96, I <= 8, and a tile of x that fits shared memory."""
    return bool(
        isinstance(gru, torch.nn.GRU) and gru.num_layers == 1 and not gru.bidirectional and gru.batch_first and gru.bias
        and getattr(gru, "proj_size", 0) == 0
        and isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 3
        and x.size(2) == gru.input_size and x.size(1) >= 1
        and all(t.device == x.device and t.dtype == torch.float32
                for t in (gru.weight_ih_l0, gru.weight_hh_l0, gru.bias_ih_l0, gru.bias_hh_l0))
        and gru.weight_hh_l0.data_ptr() % 16 == 0
        and lib.sldm_gru_supported(int(x.size(1)), int(x.size(2)), int(gru.hidden_size)))


def decode_partials(P: torch.Tensor, H: int, I: int):
    """Summed per-tile partials of sldm_gru_backward -> (dW_ih [3H,I], db_ih [3H], db_hh [3H]).

    Layout (include/sldm_sage.h): [28*U][32 lanes], U = H/32; v = (u*3+g)*8 + i -> dW_ih[g*H + 32u + lane][i];
    v = 24U + u*3 + g -> db_ih[g*H + 32u + lane]; v = 27U + u -> db_hh[2H + 32u + lane]; db_hh[:2H] = db_ih[:2H]
    (the r and z gates see the same pre-activation gradient on the input and the hidden side)."""
    U = H // 32
    dW_ih = P[:24 * U * 32].view(U, 3, 8, 32).permute(1, 0, 3, 2).reshape(3 * H, 8)[:, :I].contiguous()
    db_ih = P[24 * U * 32:27 * U * 32].view(U, 3, 32).permute(1, 0, 2).reshape(3 * H)
    db_hh = torch.cat([db_ih[:2 * H], P[27 * U * 32:]])
    return dW_ih, db_ih, db_hh


class _GruLastHiddenFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, W_ih, W_hh, b_ih, b_hh):
        N, T, I = x.shape
        H = W_hh.shape[1]
        dev = x.device
        save = any(ctx.needs_input_grad)
        x, W_ih, W_hh, b_ih, b_hh = (t.contiguous() for t in (x, W_ih, W_hh, b_ih, b_hh))
        with torch.cuda.device(dev):
            h_last = torch.empty((N, H), dtype=torch.float32, device=dev)
            saved = torch.empty((T, N, 5, H), dtype=torch.float32, device=dev) if save else None
            check(lib.sldm_gru_forward(x.data_ptr(), N, T, I, H, W_ih.data_ptr(), W_hh.data_ptr(), b_ih.data_ptr(),
                                       b_hh.data_ptr(), h_last.data_ptr(), _ptr(saved), _stream(dev)))
        if save:
            ctx.save_for_backward(x, W_ih, W_hh, saved)
        return h_last

    @staticmethod
    @once_differentiable   # hand-written first-order gradients: a double backward raises instead of returning garbage
    def backward(ctx, dh_last):
        x, W_ih, W_hh, saved = ctx.saved_tensors
        N, T, I = x.shape
        H = W_hh.shape[1]
        dev = x.device
        need_dx = ctx.needs_input_grad[0]
        dh_last = dh_last.contiguous()
        with torch.cuda.device(dev):
            f32 = dict(dtype=torch.float32, device=dev)
            dgh = torch.empty((T, N, 3 * H), **f32)
            dgi_n = torch.empty((T, N, H), **f32) if need_dx else None
            rows, width = int(lib.sldm_gru_partial_rows(N)), int(lib.sldm_gru_partial_width(H))
            parts = torch.empty((rows, width), **f32)
            check(lib.sldm_gru_backward(x.data_ptr(), N, T, I, H, W_hh.data_ptr(), dh_last.data_ptr(),
                                        saved.data_ptr(), dgh.data_ptr(), _ptr(dgi_n), parts.data_ptr(), rows,
                                        _stream(dev)))
            dW_ih, db_ih, db_hh = decode_partials(parts.sum(dim=0), H, I)
            tiles = int(lib.sldm_gru_wgrad_tiles(N, T))
            wparts = torch.empty((tiles, 3 * H, H), **f32)
            check(lib.sldm_gru_wgrad(dgh.data_ptr(), saved.data_ptr(), N, T, H, wparts.data_ptr(), tiles, _stream(dev)))
            dW_hh = wparts.sum(dim=0)
            dgh2 = dgh.view(T * N, 3 * H)
            dx = None
            if need_dx:
                dgi = torch.cat([dgh2[:, :2 * H], dgi_n.view(T * N, H)], dim=1)
                dx = (dgi @ W_ih).view(T, N, I).transpose(0, 1).contiguous()
        return dx, dW_ih, dW_hh, db_ih, db_hh


def gru_last_hidden(gru: torch.nn.GRU, x: torch.Tensor) -> torch.Tensor:
    """`gru(x)[1][-1]` with h0 = 0 for an eligible module / input (see `fused_gru_eligible`)."""
    _require_cuda(x, "x")
    if not fused_gru_eligible(gru, x):
        raise NotImplementedError("gru_last_hidden: this nn.GRU / input is outside the fused kernels' range "
                                  "(one batch-first layer, hidden 32/64/96, input width <= 8, fp32 CUDA)")
    return _GruLastHiddenFn.apply(x, gru.weight_ih_l0, gru.weight_hh_l0, gru.bias_ih_l0, gru.bias_hh_l0)


def _stack_params(gru: torch.nn.GRU):
    return [getattr(gru, f"{kind}_l{k}") for k in range(gru.num_layers)
            for kind in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]


def fused_gru_stack_eligible(gru: torch.nn.GRU, x: torch.Tensor) -> bool:
    """True when `gru(x)[1][-1]` of a (possibly) stacked nn.GRU can run on the fused kernels: unidirectional,
    batch-first, with biases, no projection, no inter-layer dropout in training, fp32 CUDA input [N, T, I], hidden
    size 32 / 64 / 96, and layer 0 within the single-layer range (I <= 8, its x tile fits shared memory); the layers
    above have no limit on T."""
    return bool(
        isinstance(gru, torch.nn.GRU) and gru.num_layers >= 1 and not gru.bidirectional and gru.batch_first and gru.bias
        and getattr(gru, "proj_size", 0) == 0 and (gru.dropout == 0 or not gru.training)
        and isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 3
        and x.size(2) == gru.input_size and x.size(1) >= 1
        and all(t.device == x.device and t.dtype == torch.float32 for t in _stack_params(gru))
        and all(getattr(gru, f"weight_hh_l{k}").data_ptr() % 16 == 0 for k in range(gru.num_layers))
        and lib.sldm_gru_stack_supported(int(x.size(1)), int(x.size(2)), int(gru.hidden_size)))


class _GruStackLastHiddenFn(torch.autograd.Function):
    """Last hidden state of the top layer of an L-layer GRU.  Launches: forward 1 + 2(L-1) (layer 0's recurrence, then
    per layer above the input projection and the recurrence), backward 2 + 4(L-1) (per layer above: the reverse
    recurrence, dW_hh, dW_ih and the projection of dgi back onto the layer below; layer 0: reverse recurrence and dW_hh;
    the layer-0 dx product is torch's, as in the single-layer path).  Every sequence buffer is time-major."""

    @staticmethod
    def forward(ctx, x, *params):
        N, T, I = x.shape
        L = len(params) // 4
        H = params[1].shape[1]
        dev = x.device
        save = any(ctx.needs_input_grad)
        x = x.contiguous()
        params = [p.contiguous() for p in params]
        saved, h_seqs = [], []
        with torch.cuda.device(dev):
            f32 = dict(dtype=torch.float32, device=dev)
            h_last = torch.empty((N, H), **f32)
            h_below = None
            for l in range(L):
                W_ih, W_hh, b_ih, b_hh = params[4 * l:4 * l + 4]
                top = l == L - 1
                s = torch.empty((T, N, 5, H), **f32) if save else None
                h_seq = None if top else torch.empty((T, N, H), **f32)
                if l == 0:
                    check(lib.sldm_gru_layer_forward(x.data_ptr(), None, N, T, I, H, W_ih.data_ptr(), W_hh.data_ptr(),
                                                     b_ih.data_ptr(), b_hh.data_ptr(), _ptr(h_last if top else None),
                                                     _ptr(s), _ptr(h_seq), _stream(dev)))
                else:
                    gi = torch.empty((T, N, 3 * H), **f32)
                    check(lib.sldm_gru_project_forward(h_below.data_ptr(), N * T, H, W_ih.data_ptr(), b_ih.data_ptr(),
                                                       gi.data_ptr(), _stream(dev)))
                    check(lib.sldm_gru_layer_forward(None, gi.data_ptr(), N, T, I, H, None, W_hh.data_ptr(), None,
                                                     b_hh.data_ptr(), _ptr(h_last if top else None), _ptr(s),
                                                     _ptr(h_seq), _stream(dev)))
                    del gi
                saved.append(s)
                if h_seq is not None:
                    h_seqs.append(h_seq)
                h_below = h_seq
        if save:
            ctx.save_for_backward(x, *params, *saved, *h_seqs)
            ctx.num_layers = L
        return h_last

    @staticmethod
    @once_differentiable   # hand-written first-order gradients: a double backward raises instead of returning garbage
    def backward(ctx, dh_last):
        L = ctx.num_layers
        x, rest = ctx.saved_tensors[0], ctx.saved_tensors[1:]
        params, saved, h_seqs = rest[:4 * L], rest[4 * L:5 * L], rest[5 * L:]
        N, T, I = x.shape
        H = params[1].shape[1]
        dev = x.device
        need_dx = ctx.needs_input_grad[0]
        dh_last = dh_last.contiguous()
        grads = [None] * (4 * L)
        dx = None
        with torch.cuda.device(dev):
            f32 = dict(dtype=torch.float32, device=dev)
            rows, width = int(lib.sldm_gru_partial_rows(N)), int(lib.sldm_gru_partial_width(H))
            tiles = int(lib.sldm_gru_wgrad_tiles(N, T))
            dy = None                       # gradient of h^l_t from the layer above, [T,N,H]
            for l in range(L - 1, -1, -1):
                W_ih, W_hh = params[4 * l], params[4 * l + 1]
                top, deep = l == L - 1, l > 0
                dgh = torch.empty((T, N, 3 * H), **f32)
                dgi = torch.empty((T, N, 3 * H), **f32) if deep else None
                dgi_n = torch.empty((T, N, H), **f32) if not deep and need_dx else None
                parts = torch.empty((rows, width), **f32)
                check(lib.sldm_gru_layer_backward(None if deep else x.data_ptr(), N, T, I, H, W_hh.data_ptr(),
                                                  _ptr(dh_last if top else None), _ptr(dy), saved[l].data_ptr(),
                                                  dgh.data_ptr(), _ptr(dgi_n), _ptr(dgi), parts.data_ptr(), rows,
                                                  _stream(dev)))
                dW_ih, db_ih, db_hh = decode_partials(parts.sum(dim=0), H, 1 if deep else I)
                wparts = torch.empty((tiles, 3 * H, H), **f32)
                check(lib.sldm_gru_wgrad(dgh.data_ptr(), saved[l].data_ptr(), N, T, H, wparts.data_ptr(), tiles,
                                         _stream(dev)))
                dW_hh = wparts.sum(dim=0)
                if deep:
                    check(lib.sldm_gru_wgrad_strided(dgi.data_ptr(), h_seqs[l - 1].data_ptr(), H, N, T, H,
                                                     wparts.data_ptr(), tiles, _stream(dev)))
                    dW_ih = wparts.sum(dim=0)
                    dy = torch.empty((T, N, H), **f32)
                    check(lib.sldm_gru_project_backward(dgi.data_ptr(), N * T, H, W_ih.data_ptr(), dy.data_ptr(),
                                                        _stream(dev)))
                elif need_dx:
                    dgh2 = dgh.view(T * N, 3 * H)
                    dgi0 = torch.cat([dgh2[:, :2 * H], dgi_n.view(T * N, H)], dim=1)
                    dx = (dgi0 @ W_ih).view(T, N, I).transpose(0, 1).contiguous()
                grads[4 * l:4 * l + 4] = [dW_ih, dW_hh, db_ih, db_hh]
        return (dx, *grads)


def gru_stack_last_hidden(gru: torch.nn.GRU, x: torch.Tensor) -> torch.Tensor:
    """`gru(x)[1][-1]` with h0 = 0 for an eligible (possibly stacked) module / input (see `fused_gru_stack_eligible`)."""
    _require_cuda(x, "x")
    if not fused_gru_stack_eligible(gru, x):
        raise NotImplementedError("gru_stack_last_hidden: this nn.GRU / input is outside the fused kernels' range "
                                  "(batch-first unidirectional layers, hidden 32/64/96, input width <= 8, fp32 CUDA, "
                                  "no inter-layer dropout in training)")
    return _GruStackLastHiddenFn.apply(x, *_stack_params(gru))
