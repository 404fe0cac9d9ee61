"""The model around the block: GruSage, MapEncoder, MapZscoreNorm as drop-ins composed of this package's kernels.

Reference: src/models/grusage.py:12-215 (GruSage), src/models/map/mapencoder.py:6-38 (MapEncoder),
src/models/map/mapInputNorm.py:3-23 (MapZscoreNorm).  This is SURVEY 8(d)'s configuration C2 -- the full training step
of the reference's model in an image without torch_geometric: the graph layers (SageBlock, twice: map graph and vehicle
graph), the map attention and the readout are the CUDA paths of libsldm_sage.so; the station-type embedding, the GRU and
the small fully connected stacks are torch library layers, as in the reference (the GRU through ATen's native cuBLAS
path instead of cuDNN: 3.3x faster at this shape and true fp32, see GruSage._last_hidden).

Same constructor arguments, same module tree (`st_emb`, `gru`, `fc1s`, `map_encoder`, `map_attention`, `sage`, `fc2s`,
`linout`), so the reference's checkpoints load strictly and `state_dict_no_mapenc()` / `input_params_dict()` /
`grads()` keep their meaning.  `forward(data)` reads the same attributes of a PyG Batch (or of our GraphBatch):
x [N,T,F], edge_index, xsttype, xdims, pos_raw, batch.  Differences, both invisible in the results:
  * 'double' pooling is ONE fused mean|max readout kernel instead of two pools and a cat;
  * the number of graphs is taken from `data.num_graphs` when the batch carries it (PyG reads `batch.max()` back from
    the device, a host sync per step).
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn

from .gru import (fused_gru_eligible, fused_gru_projected_eligible, fused_gru_stack_eligible, gru_last_hidden,
                  gru_projected_last_hidden, gru_stack_last_hidden)
from .map_attention import MapSpatialAttention
from .ops import index_checks
from .readout import global_max_pool, global_mean_max_pool, global_mean_pool
from .sageblock import SageBlock


def _activation(negative_slope):
    return nn.ReLU() if negative_slope is None else nn.LeakyReLU(negative_slope=negative_slope)


def _fc_stack(widths, dropout, negative_slope) -> nn.ModuleList:
    """Linear -> (Leaky)ReLU -> Dropout|Identity per consecutive pair of widths (grusage.py:63-70, 132-138)."""
    return nn.ModuleList(
        nn.Sequential(nn.Linear(a, b), _activation(negative_slope), nn.Identity() if dropout is None else nn.Dropout(p=dropout))
        for a, b in zip(widths[:-1], widths[1:]))


class MapZscoreNorm:
    """Per-feature z-score over the segments, population variance, sigma clamped at 1e-8 (mapInputNorm.py:12-23)."""

    def __init__(self, map_float_features: torch.Tensor):
        n = map_float_features.shape[0]
        self.mu = map_float_features.sum(dim=0, keepdim=True) / n
        self.sigma = (((map_float_features - self.mu) ** 2).sum(dim=0, keepdim=True) / n).sqrt().clamp(min=1e-8)

    def __call__(self, map_input: torch.Tensor) -> torch.Tensor:
        return (map_input - self.mu) / self.sigma

    @classmethod
    def onfly(cls, map_float_features: torch.Tensor) -> torch.Tensor:
        return cls(map_float_features)(map_float_features)


class MapEncoder(nn.Module):
    """Embeds the static map graph: [float | bool | lane-type embedding] features through a SageBlock
    (mapencoder.py:6-38).  The map's edge_index is a buffer that never changes, so the block's CSR cache builds its CSR
    once and every later step is gather + projection only."""

    def __init__(self, map_float_features, map_bool_features, lane_type_cats, graph_edge_indexes, *, lane_embed_dim=2,
                 sage_hidden_dims=[8, 8], dropout, negative_slope):
        super().__init__()
        feats = torch.cat([map_float_features, map_bool_features.to(map_float_features.dtype)], dim=1)
        self.register_buffer("map_float_features", feats, persistent=False)
        self.register_buffer("lane_type_cats", lane_type_cats, persistent=False)
        self.register_buffer("graph_edge_indexes", graph_edge_indexes, persistent=False)
        self.lane_embedding = nn.Embedding(int(lane_type_cats.max().item()) + 1, lane_embed_dim)
        self.sage = SageBlock([feats.shape[1] + lane_embed_dim] + list(sage_hidden_dims), dropout=dropout,
                              negative_slope=negative_slope)
        self._out_dim = sage_hidden_dims[-1]

    @property
    def out_dim(self) -> int:
        return self._out_dim

    def forward(self) -> torch.Tensor:
        x = torch.cat([self.map_float_features, self.lane_embedding(self.lane_type_cats)], dim=1)
        return self.sage(x, self.graph_edge_indexes)


_POOLS = {"mean": (global_mean_pool, 1), "max": (global_max_pool, 1), "double": (global_mean_max_pool, 2)}


class GruSage(nn.Module):
    def __init__(self, dynamic_features_num, frames_num, gru_hidden_size, gru_num_layers, fc1dims, sage_hidden_dims=[128, 128],
                 fc2dims=[50, 50], out_dim=1, num_st_types=256, emb_dim=12, dropout=None, negative_slope=None,
                 global_pooling="double", map_included=True, *, map_tensors=None, mapenc_sage_hdims=[8, 8],
                 mapenc_lane_embdim=2, map_attention_topk=5, map_embeddings=None, map_centroids=None):
        super().__init__()
        if map_included:        # grusage.py:16-20
            assert (map_tensors is not None) or (map_embeddings is not None), \
                "If map_included is True, either map_tensors or map_embeddings must be provided"
            assert map_attention_topk is not None, "If map_included is True, map_attention_topk must be provided"
            assert (map_tensors is None) or (map_embeddings is None), "Provide either map_tensors or map_embeddings, not both"
            assert (map_embeddings is None) == (map_centroids is None), \
                "If providing map_embeddings directly, also provide map_centroids for attention"
        assert len(sage_hidden_dims) >= 1, "sage_hidden_dims must contain at least one element"
        if global_pooling not in _POOLS:
            raise ValueError(f"Unsupported global_pooling method: {global_pooling}")
        # the snapshot of the constructor arguments (grusage.py:23-42; the map tensors come back through the state dict)
        self.config_dict = dict(
            dynamic_features_num=dynamic_features_num, frames_num=frames_num, gru_hidden_size=gru_hidden_size,
            gru_num_layers=gru_num_layers, fc1dims=fc1dims, sage_hidden_dims=sage_hidden_dims, fc2dims=fc2dims, out_dim=out_dim,
            num_st_types=num_st_types, emb_dim=emb_dim, dropout=dropout, negative_slope=negative_slope,
            global_pooling=global_pooling, map_included=map_included, map_attention_topk=map_attention_topk,
            map_embeddings=map_embeddings, map_centroids=map_centroids)
        self.dropout, self.negative_slope = dropout, negative_slope

        self.st_emb = nn.Embedding(num_st_types, emb_dim)
        self.gru = nn.GRU(input_size=dynamic_features_num, hidden_size=gru_hidden_size, num_layers=gru_num_layers, batch_first=True)
        width = gru_hidden_size + 2 + emb_dim                       # last hidden state | xdims | station-type embedding
        self.fc1s = _fc_stack([width] + list(fc1dims), dropout, negative_slope)
        width = ([width] + list(fc1dims))[-1]

        # NOTE the reference only defines these two attributes when map_included is True (grusage.py:74-76) and its
        # forward() reads map_provided unconditionally; here they always exist
        self.map_provided = bool(map_included)
        self.map_tensors = map_included and map_tensors is not None
        if map_included:
            if map_tensors is not None:
                self.map_encoder = MapEncoder(
                    map_float_features=MapZscoreNorm.onfly(map_tensors["float_features"]),
                    map_bool_features=map_tensors["bool_features"], lane_type_cats=map_tensors["lane_type_cats"],
                    graph_edge_indexes=map_tensors["mgraph_edge_indexes"], lane_embed_dim=mapenc_lane_embdim,
                    sage_hidden_dims=mapenc_sage_hdims, dropout=dropout, negative_slope=negative_slope)
                self.map_attention = MapSpatialAttention(map_centroids=map_tensors["mseg_centroids"], k_neighbors=map_attention_topk)
                width += self.map_encoder.out_dim
            else:
                self.register_buffer("map_embeddings", map_embeddings, persistent=False)
                self.map_attention = MapSpatialAttention(map_centroids=map_centroids, k_neighbors=map_attention_topk)
                width += map_embeddings.shape[1]

        self.sage = SageBlock([width] + list(sage_hidden_dims), dropout=dropout, negative_slope=negative_slope)
        self._pool, mult = _POOLS[global_pooling]
        self.fc2s = _fc_stack([sage_hidden_dims[-1] * mult] + list(fc2dims), dropout, negative_slope)
        self.linout = nn.Linear(([sage_hidden_dims[-1] * mult] + list(fc2dims))[-1], out_dim)

    # the reference exposes the pooling as an attribute (grusage.py:113-120)
    def global_pool(self, x, batch, size=None):
        return self._pool(x, batch, size)

    def state_dict_no_mapenc(self):
        return {k: v for k, v in self.state_dict().items() if not k.startswith("map_encoder")}

    def input_params_dict(self):
        ipd = dict(self.config_dict)
        with torch.no_grad():
            ipd["map_embeddings"] = (self.map_encoder() if self.map_tensors else self.map_embeddings) if self.map_provided else None
            ipd["map_centroids"] = self.map_attention.map_centroids if self.map_provided else None
        return ipd

    def _last_hidden(self, x):
        """[N, T, F] -> last hidden state of the last GRU layer (grusage.py:160-161).

        Default: the fused kernels of csrc/gru.cu (all T steps of a tile of sequences on one SM; gru.py) whenever the
        module is one batch-first layer with hidden 32 / 64 / 96 and at most 8 input features -- the reference's
        configuration (main.py:42-44: hidden 96, one layer, 6 dynamic features).  A stacked head (gru_num_layers > 1)
        with the same limits on its first layer runs on the same kernels layer by layer (gru_stack_last_hidden: the
        layers above take their input projection from k_gru_proj and have no limit on T), unless inter-layer dropout
        is active in training.  Sequences too long or inputs too wide for layer 0's x tile (for example more than 30
        frames at hidden 96, or more than 8 dynamic features) take the projected path (gru_projected_last_hidden: x is
        first projected into the gate pre-activations gi by k_gru_xproj, up to 128 features, any number of frames).
        The tile is preferred wherever it applies, since it saves gi's round trip through HBM; the choice follows from
        the shape alone.  Anything else, or SLDM_DISABLE_FUSED_GRU=1, goes through torch's library GRU, and there through ATen's native path (one cuBLAS
        GEMM + one fused cell kernel per step) rather than cuDNN's: measured on B200 at the C2 shape (205 k sequences
        x 16 frames, input 6, hidden 96) the native path takes 35 ms forward + backward against 118 ms, and it computes
        in true fp32 -- cuDNN's RNN runs TF32 under torch's default flags (2e-4 off the CPU result,
        tools/gru_probe.py), which is outside this package's 1e-5 bar.  cuDNN also indexes its gate workspace
        (N * T * 3H elements) with 32 bits and faults beyond 2^31; sequences are independent, so very large batches go
        through the library path in slices -- same numbers, no limit."""
        if os.environ.get("SLDM_DISABLE_FUSED_GRU", "0") != "1":
            if fused_gru_eligible(self.gru, x):
                return gru_last_hidden(self.gru, x)
            if fused_gru_stack_eligible(self.gru, x):
                return gru_stack_last_hidden(self.gru, x)
            if fused_gru_projected_eligible(self.gru, x):
                return gru_projected_last_hidden(self.gru, x)
        n, per_seq = x.size(0), x.size(1) * 3 * self.gru.hidden_size
        rows = max(1, (1 << 30) // max(per_seq, 1))
        with torch.backends.cudnn.flags(enabled=False):
            if n <= rows:
                return self.gru(x)[1][-1]
            return torch.cat([self.gru(x[i:i + rows])[1][-1] for i in range(0, n, rows)], dim=0)

    def forward(self, data):
        h = self._last_hidden(data.x)
        x = torch.cat([h, data.xdims, self.st_emb(data.xsttype)], dim=1)
        for fc in self.fc1s:
            x = fc(x)
        if self.map_provided:
            emb = self.map_encoder() if self.map_tensors else self.map_embeddings
            ctx = self.map_attention(vehicle_last_positions=data.pos_raw[:, -1, :], map_embeddings=emb)
            x = torch.cat([x, ctx], dim=1)
        x = self.sage(x, data.edge_index)
        x = self._pool(x, data.batch, getattr(data, "num_graphs", None))
        for fc in self.fc2s:
            x = fc(x)
        return self.linout(x)

    def grads(self):
        """Gradient norms per group of layers and in total (grusage.py:197-215)."""
        groups = {"StType Embedding": self.st_emb, "GRU Layer": self.gru, "FC Layers before SAGE": self.fc1s,
                  "GraphSAGE Layers": self.sage, "FC Layers after SAGE": self.fc2s, "Final Output Layer": self.linout}
        flat = {}
        for name, module in groups.items():
            parts = [p.grad.view(-1) for p in module.parameters() if p.requires_grad and p.grad is not None]
            flat[name] = torch.cat(parts) if parts else None
        present = [g for g in flat.values() if g is not None]
        total = torch.cat(present).norm().item() if present else None
        return total, {name: (g.norm().item() if g is not None else None) for name, g in flat.items()}


class _TensorArgs(nn.Module):
    """GruSage.forward over plain tensors (torch.cuda.make_graphed_callables wants tensor arguments)."""

    def __init__(self, model: "GruSage", num_graphs: int):
        super().__init__()
        self.model, self.num_graphs = model, int(num_graphs)

    def forward(self, x, xdims, xsttype, pos_raw, edge_index, batch):
        from types import SimpleNamespace
        self.model.sage.clear_cache()      # inside a CUDA graph the CSR build of the batch must be part of every replay
        out = self.model(SimpleNamespace(x=x, xdims=xdims, xsttype=xsttype, pos_raw=pos_raw, edge_index=edge_index,
                                         batch=batch, num_graphs=self.num_graphs))
        self.model.sage.clear_cache()
        return out


class GraphedGruSage:
    """GruSage.forward (+ its backward) through captured CUDA graphs for batches of up to max_nodes - 1 vehicles,
    max_edges edges and max_graphs - 1 graphs -- the reference trains on batches of 32 graphs (main.py:24) and tests on
    64 (test.py:58), where the ~200 kernel launches of a step and their Python glue cost several times the kernels.

        g = GraphedGruSage(model, max_nodes=8192, max_edges=40960, max_graphs=33)
        loss = crit(g(data), data.y); loss.backward(); opt.step()      # forward graph + backward graph, autograd-aware

    The captured step works on static buffers of the bucket's size.  Rows [0, N) hold the batch; the padding vehicles
    [N, max_nodes) belong to one extra padding graph (id max_graphs - 1), the padding edges are self loops of the last
    padding vehicle.  Every stage is row-wise independent (GRU, fc stacks, map attention, SageBlock) or graph-wise
    independent (readout), so the logits of the real graphs see the same inputs as in the un-captured model; the
    padding graph's logit is sliced off, its upstream gradient is exactly zero and the parameter gradients therefore
    equal the un-captured ones up to the association of their fp32 sums.  training=True uses
    torch.cuda.make_graphed_callables (dropout draws from the graph-safe generator state); training=False captures one
    inference graph (eval mode).  The returned logits are a view of the graph's static output, valid until the next
    call.  Thread-safe: calls serialise on a lock.  Like any use of make_graphed_callables, construct it while no
    autograd graph of an earlier eager step of the same model is alive (a kept `loss` is enough): the backward capture
    would have to synchronise with the default stream and is invalidated.
    """

    _FIELDS = ("x", "xdims", "xsttype", "pos_raw", "edge_index", "batch")

    def __init__(self, model: "GruSage", max_nodes: int, max_edges: int, max_graphs: int, training: bool = True):
        import threading
        p0 = next(model.parameters())
        if p0.device.type != "cuda":
            raise RuntimeError("GraphedGruSage: CUDA only")
        self.model, self.dev, self.training = model, p0.device, bool(training)
        self.max_nodes, self.max_edges, self.max_graphs = int(max_nodes), int(max_edges), int(max_graphs)
        cfg = model.config_dict
        T, F = int(cfg["frames_num"]), int(cfg["dynamic_features_num"])
        dev, Nm, Em = self.dev, self.max_nodes, self.max_edges
        self._lock = threading.Lock()
        with torch.cuda.device(dev):
            self._static = dict(
                x=torch.zeros((Nm, T, F), device=dev), xdims=torch.zeros((Nm, 2), device=dev),
                xsttype=torch.zeros((Nm,), dtype=torch.long, device=dev), pos_raw=torch.zeros((Nm, T, 2), device=dev),
                edge_index=torch.full((2, Em), Nm - 1, dtype=torch.long, device=dev),
                batch=torch.full((Nm,), self.max_graphs - 1, dtype=torch.long, device=dev))
            args = tuple(self._static[k] for k in self._FIELDS)
            wrapped = _TensorArgs(model, self.max_graphs)
            index_checks.poll(block=True)                      # nothing may be pending when a capture starts
            if self.training:
                model.train()
                self._call = torch.cuda.make_graphed_callables(wrapped, args, allow_unused_input=True)
            else:
                was_training = model.training
                model.eval()
                with torch.inference_mode():
                    side = torch.cuda.Stream(device=dev)
                    side.wait_stream(torch.cuda.current_stream(dev))
                    with torch.cuda.stream(side):              # warm-up outside the capture: opt-in attributes, caches
                        for _ in range(2):
                            wrapped(*args)
                    torch.cuda.current_stream(dev).wait_stream(side)
                    torch.cuda.synchronize(dev)
                    index_checks.poll(block=True)
                    self._graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(self._graph):
                        self._y = wrapped(*args)
                model.train(was_training)
            # objects the captured kernels read but the graph does not own: the static map graph's CSR and the
            # centroid grid of the attention stay alive as long as this object does
            self._keep = []
            if getattr(model, "map_tensors", False):
                self._keep.append(model.map_encoder.sage._csr)
            if getattr(model, "map_provided", False):
                self._keep.append((model.map_attention._grid, getattr(model.map_attention, "_grid_cent", None)))

    def _fill(self, data, N, E):
        s = self._static
        with torch.no_grad():
            s["x"][:N].copy_(data.x, non_blocking=True)
            s["xdims"][:N].copy_(data.xdims, non_blocking=True)
            s["xsttype"][:N].copy_(data.xsttype, non_blocking=True)
            s["pos_raw"][:N].copy_(data.pos_raw, non_blocking=True)
            s["batch"][:N].copy_(data.batch, non_blocking=True)
            s["batch"][N:].fill_(self.max_graphs - 1)
            s["edge_index"][:, :E].copy_(data.edge_index, non_blocking=True)
            if E < self.max_edges:
                s["edge_index"][:, E:].fill_(self.max_nodes - 1)
        # feature rows beyond N keep what an earlier, larger batch left there: they are padding vehicles now (no edge
        # from a real vehicle reaches them, they pool into the padding graph), so their values never matter

    def __call__(self, data) -> torch.Tensor:
        N, E = int(data.x.size(0)), int(data.edge_index.size(1))
        G = getattr(data, "num_graphs", None)
        if G is None:
            raise RuntimeError("GraphedGruSage: data.num_graphs is required (reading it off `batch` would synchronise)")
        if N >= self.max_nodes or E > self.max_edges or G >= self.max_graphs:
            raise RuntimeError(f"GraphedGruSage: N = {N}, E = {E}, graphs = {G} exceed the bucket ({self.max_nodes - 1} vehicles, "
                               f"{self.max_edges} edges, {self.max_graphs - 1} graphs)")
        with self._lock, torch.cuda.device(self.dev):
            self._fill(data, N, E)
            if self.training:
                return self._call(*(self._static[k] for k in self._FIELDS))[:G]
            self._graph.replay()
            return self._y[:G].clone()


class GraphedTrainStep:
    """One whole training step of a GruSage -- zero_grad, forward, loss, backward, optimizer step (the body of the
    reference's loop, src/utils.py:218-236) -- as ONE captured CUDA graph over the padded static buffers of
    GraphedGruSage: per step the host copies the batch in, launches one graph and reads the loss.

        opt  = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=5e-5, capturable=True)   # fused=True works too
        step = GraphedTrainStep(model, opt, loss_fn, max_nodes=8192, max_edges=40960, max_graphs=33)
        loss = step(data, data.y)            # 0-dim device tensor (static: valid until the next call); .item() to read it

    loss_fn(logits [max_graphs, out], y [max_graphs, out], weight [max_graphs, 1]) -> scalar must be a weighted SUM:
    `weight` is 1 / num_graphs on the rows of real graphs and 0 on the padding rows, so that e.g.
    F.binary_cross_entropy_with_logits(logits, y, weight=weight, pos_weight=pw, reduction="sum") is the reference's
    BCEWithLogitsLoss(pos_weight) mean over the real graphs.  The optimizer must be capturable (its step counter lives
    on the device).  Warm-up and capture run the step on all-padding inputs; parameters and optimizer state are put back
    in place afterwards (state tensors the optimizer created during warm-up are zeroed: Adam / AdamW / SGD momentum).
    After a call every parameter's .grad holds this step's gradient (the reference logs gradient norms from it).
    """

    def __init__(self, model: "GruSage", optimizer, loss_fn, max_nodes: int, max_edges: int, max_graphs: int):
        import threading
        if not all(g.get("capturable", False) for g in optimizer.param_groups):
            raise ValueError("GraphedTrainStep: the optimizer must be constructed with capturable=True")
        base = GraphedGruSage.__new__(GraphedGruSage)          # static buffers and padding rules are GraphedGruSage's
        p0 = next(model.parameters())
        if p0.device.type != "cuda":
            raise RuntimeError("GraphedTrainStep: CUDA only")
        base.model, base.dev, base.training = model, p0.device, True
        base.max_nodes, base.max_edges, base.max_graphs = int(max_nodes), int(max_edges), int(max_graphs)
        cfg = model.config_dict
        T, F, out_dim = int(cfg["frames_num"]), int(cfg["dynamic_features_num"]), int(cfg["out_dim"])
        dev, Nm, Em, Gm = base.dev, base.max_nodes, base.max_edges, base.max_graphs
        self._base, self.model, self.dev, self._lock = base, model, dev, threading.Lock()
        with torch.cuda.device(dev):
            base._static = dict(
                x=torch.zeros((Nm, T, F), device=dev), xdims=torch.zeros((Nm, 2), device=dev),
                xsttype=torch.zeros((Nm,), dtype=torch.long, device=dev), pos_raw=torch.zeros((Nm, T, 2), device=dev),
                edge_index=torch.full((2, Em), Nm - 1, dtype=torch.long, device=dev),
                batch=torch.full((Nm,), Gm - 1, dtype=torch.long, device=dev))
            self._y = torch.zeros((Gm, out_dim), device=dev)
            self._w = torch.zeros((Gm, 1), device=dev)
            args = tuple(base._static[k] for k in GraphedGruSage._FIELDS)
            wrapped = _TensorArgs(model, Gm)
            params = [p for g in optimizer.param_groups for p in g["params"]]
            saved_p = [p.detach().clone() for p in params]
            had_state = {id(p): {k: (v.detach().clone() if torch.is_tensor(v) else v) for k, v in optimizer.state.get(p, {}).items()}
                         for p in params}
            model.train()

            def one_step():
                optimizer.zero_grad(set_to_none=True)
                loss = loss_fn(wrapped(*args), self._y, self._w)
                loss.backward()
                optimizer.step()
                return loss

            index_checks.poll(block=True)                      # nothing may be pending when a capture starts
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(3):
                    one_step()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            index_checks.poll(block=True)
            optimizer.zero_grad(set_to_none=True)
            self._graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._graph):
                self._loss = one_step()
            torch.cuda.synchronize(dev)
            self._params, self._grads = params, [p.grad for p in params]   # the graph's static gradient tensors
            with torch.no_grad():                              # undo the warm-up steps, in place (the graph holds the pointers)
                for p, s in zip(params, saved_p):
                    p.copy_(s)
                    before = had_state[id(p)]
                    for k, v in optimizer.state.get(p, {}).items():
                        if torch.is_tensor(v):
                            v.copy_(before[k]) if k in before else v.zero_()
            base._keep = []
            if getattr(model, "map_tensors", False):
                base._keep.append(model.map_encoder.sage._csr)
            if getattr(model, "map_provided", False):
                base._keep.append((model.map_attention._grid, getattr(model.map_attention, "_grid_cent", None)))

    def __call__(self, data, y: torch.Tensor) -> torch.Tensor:
        b = self._base
        N, E = int(data.x.size(0)), int(data.edge_index.size(1))
        G = int(y.size(0))
        if N >= b.max_nodes or E > b.max_edges or G >= b.max_graphs:
            raise RuntimeError(f"GraphedTrainStep: N = {N}, E = {E}, graphs = {G} exceed the bucket ({b.max_nodes - 1} vehicles, "
                               f"{b.max_edges} edges, {b.max_graphs - 1} graphs)")
        with self._lock, torch.cuda.device(self.dev):
            b._fill(data, N, E)
            with torch.no_grad():
                self._y[:G].copy_(y, non_blocking=True)
                self._w[:G].fill_(1.0 / max(G, 1))
                self._w[G:].zero_()
            self._graph.replay()
            for p, g in zip(self._params, self._grads):        # a zero_grad(set_to_none=True) outside must not hide them
                p.grad = g
            return self._loss
