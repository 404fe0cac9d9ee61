"""Drop-in MapSpatialAttention (reference: src/models/map/mapattention.py:5-56, used at src/models/grusage.py:100-103,175-178).

Same constructor `(map_centroids, k_neighbors=5)`, same `forward(vehicle_last_positions, map_embeddings)`, same module
tree (`attn_mlp` = Sequential(Linear(1,16), ReLU, Linear(16,1)); `map_centroids` a non-persistent buffer), so the
reference's state dicts load strictly.  The arithmetic is one fused kernel of libsldm_sage.so (no [B,S] intermediates)
with a hand-written backward for the embeddings and the MLP; positions and centroids are data and get no gradient.
Distance ties are broken towards the lower segment index.  CUDA only.  k_neighbors may be 1..32
(sldm_map_attention_max_k()); up to 8 the kernels keep per-thread lists, above 8 one warp works on each position, with
the same results contract.  A larger k raises NotImplementedError.

The centroids are a constant of the module, so they are binned once into a uniform grid (sldm_map_grid_build) and every
forward is a ring search over ~40 candidates per position instead of a scan of all S; the grid is rebuilt when the
buffer is replaced, moved or written in place.  SLDM_MAP_ATTENTION_SCAN=1 selects the exhaustive kernel (same bits).
"""
from __future__ import annotations

import os

import torch
from torch.autograd.function import once_differentiable
import torch.nn as nn

from . import _lib
from ._lib import lib, check
from .ops import Csr, _ptr, _require_cuda, _stream


class _MapAttentionFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, centroids, emb, W1, b1, W2, b2, K, grid=None):
        B, S, D, H = pos.size(0), centroids.size(0), emb.size(1), W1.numel()
        dev = pos.device
        with torch.cuda.device(dev):
            out = torch.empty((B, D), dtype=torch.float32, device=dev)
            idx = torch.empty((B, K), dtype=torch.long, device=dev)
            dist = torch.empty((B, K), dtype=torch.float32, device=dev)
            w = torch.empty((B, K), dtype=torch.float32, device=dev)
            if grid is not None:
                check(lib.sldm_map_attention_forward_grid(_ptr(pos), B, grid.data_ptr(), grid.numel(), S, _ptr(emb), D, K,
                                                          _ptr(W1), _ptr(b1), _ptr(W2), _ptr(b2), H, _ptr(out), _ptr(idx),
                                                          _ptr(dist), _ptr(w), _stream(dev)))
            else:
                check(lib.sldm_map_attention_forward(_ptr(pos), B, _ptr(centroids), S, _ptr(emb), D, K, _ptr(W1), _ptr(b1),
                                                     _ptr(W2), _ptr(b2), H, _ptr(out), _ptr(idx), _ptr(dist), _ptr(w), _stream(dev)))
        if any(ctx.needs_input_grad):
            ctx.save_for_backward(emb, idx, dist, w, W1, b1, W2)
            ctx.S, ctx.K = S, K
        return out

    @staticmethod
    @once_differentiable   # hand-written first-order gradients: a double backward raises instead of returning garbage
    def backward(ctx, dout):
        emb, idx, dist, w, W1, b1, W2 = ctx.saved_tensors
        B, K, S, D, H = idx.size(0), ctx.K, ctx.S, emb.size(1), W1.numel()
        dev = emb.device
        dout = dout.contiguous()
        need_emb = ctx.needs_input_grad[2]
        with torch.cuda.device(dev):
            demb = torch.empty_like(emb) if need_emb else None
            dW1, db1, dW2 = (torch.empty_like(W1), torch.empty_like(b1), torch.empty_like(W2))
            db2 = torch.empty((1,), dtype=torch.float32, device=dev)
            csr_buf, nodes = None, max(S, 1)
            if need_emb and B > 0:                          # (vehicle, k) pairs grouped by selected segment, in order
                layout = _lib.csr_layout(nodes, B * K)
                csr_buf = torch.empty(layout["total"], dtype=torch.int32, device=dev)
                wsb = int(lib.sldm_csr_workspace_bytes(nodes, B * K))
                ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
                check(lib.sldm_csr_build_pairs(None, idx.data_ptr(), B * K, nodes, csr_buf.data_ptr(), ws.data_ptr(), wsb, _stream(dev)))
            wsb2 = int(lib.sldm_map_attention_workspace_bytes_k(B, H, K))
            ws2 = torch.empty(max(wsb2, 1), dtype=torch.uint8, device=dev)
            check(lib.sldm_map_attention_backward(_ptr(dout), B, _ptr(emb), S, D, K, _ptr(idx), _ptr(dist), _ptr(w),
                                                  _ptr(W1), _ptr(b1), _ptr(W2), H, _ptr(csr_buf), nodes,
                                                  _ptr(demb) if (need_emb and B > 0) else None, _ptr(dW1), _ptr(db1), _ptr(dW2), _ptr(db2),
                                                  ws2.data_ptr(), wsb2, _stream(dev)))
            if need_emb and B == 0:
                demb.zero_()
        return None, None, demb, dW1, db1, dW2, db2, None, None


class MapSpatialAttention(nn.Module):
    def __init__(self, map_centroids: torch.Tensor, k_neighbors=5):
        super().__init__()
        self.register_buffer("map_centroids", map_centroids, persistent=False)
        self.k = k_neighbors
        self.attn_mlp = nn.Sequential(nn.Linear(1, 16), nn.ReLU(), nn.Linear(16, 1))
        self._grid, self._grid_key = None, None

    def _centroid_grid(self):
        """(fp32 contiguous centroids, uniform grid over them): built on first use and whenever the REGISTERED buffer
        changes (new tensor, new device, in-place write).  The cache is keyed on the buffer itself, not on a converted
        temporary -- under torch.inference_mode() (test.py:136, rcv.py:80) a temporary is an inference tensor without
        a version counter and would never match."""
        buf = self.map_centroids
        try:
            version = buf._version
        except RuntimeError:               # the buffer itself is an inference tensor: rebuild every call
            version = None
        key = (buf.data_ptr(), version, buf.size(0), buf.device, buf.dtype)
        if self._grid is None or version is None or self._grid_key != key:
            cent = buf.detach().float().contiguous()       # converted once, kept beside the grid
            S, dev = cent.size(0), cent.device
            nbytes = int(lib.sldm_map_grid_bytes(S))
            with torch.cuda.device(dev):
                grid = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                check(lib.sldm_map_grid_build(_ptr(cent), S, grid.data_ptr(), nbytes, _stream(dev)))
            self._grid, self._grid_key, self._grid_cent, self._grid_src = grid, key, cent, buf
        return self._grid_cent, self._grid

    def forward(self, vehicle_last_positions, map_embeddings):
        pos, emb, cent = vehicle_last_positions, map_embeddings, self.map_centroids
        _require_cuda(pos, "vehicle_last_positions")
        _require_cuda(emb, "map_embeddings")
        _require_cuda(cent, "map_centroids")
        if pos.dim() != 2 or pos.size(1) != 2 or cent.dim() != 2 or cent.size(1) != 2 or emb.dim() != 2:
            raise RuntimeError("MapSpatialAttention: expected positions [B,2], centroids [S,2], embeddings [S,D]")
        if emb.size(0) != cent.size(0):
            raise RuntimeError(f"MapSpatialAttention: {cent.size(0)} centroids but {emb.size(0)} embeddings")
        if cent.size(0) < self.k:
            raise RuntimeError("selected index k out of range")      # torch.topk's error
        l1, l2 = self.attn_mlp[0], self.attn_mlp[2]
        for name, t in (("attn_mlp.0.weight", l1.weight), ("attn_mlp.0.bias", l1.bias), ("attn_mlp.2.weight", l2.weight),
                        ("attn_mlp.2.bias", l2.bias)):
            if t.dtype != torch.float32 or t.device != pos.device:     # raw fp32 pointers go to the kernels
                raise RuntimeError(f"MapSpatialAttention: parameter {name} is {t.dtype} on {t.device}; expected float32 on {pos.device}")
        if os.environ.get("SLDM_MAP_ATTENTION_SCAN") == "1":
            cent, grid = cent.float().contiguous(), None
        else:
            cent, grid = self._centroid_grid()
        return _MapAttentionFn.apply(pos.float().contiguous(), cent, emb.float().contiguous(),
                                     l1.weight.reshape(-1).contiguous(), l1.bias.contiguous(),
                                     l2.weight.reshape(-1).contiguous(), l2.bias.contiguous(), int(self.k), grid)
