#!/usr/bin/env python
"""SURVEY 8(d) configuration C2: the reference's full training step (GruSage + BCEWithLogits(pos_weight) + Adam,
src/utils.py:176-236) with the graph layers, map attention and readout on this package's kernels.

    python bench.py --workload c2 [--c2-graphs 1024] [--gpus N --steps K --warmup W]      (dispatches here)

Model = the reference's default hyper-parameters (main.py:25-54): hidden 96, one GRU layer, fc1 [96], SageBlock
[128, 96, 96] (96 + 32 map context), 'double' pooling, fc2 [32], station-type embedding 8 of 256, dropout 0.25, leaky
slope 0.1, map encoder SageBlock [f+8, 32, 32] over a 2048-segment map graph, attention top-5, Adam lr 1e-3 wd 5e-5.
Batch = G sequences, each one unit vehicle graph (~200 nodes, ~1000 edges) with x [n, 16 frames, 6 features].
A step = zero_grad, forward, loss, backward, (gradient all-reduce at N > 1,) Adam step, loss.item() -- as in the
reference's loop.  value = graphs (sequences) per second over all ranks; e2e adds the per-step H2D copy of the batch from
pinned memory.  The GRU runs on the fused kernels of csrc/gru.cu (SLDM_DISABLE_FUSED_GRU=1: torch's library GRU); the
Linear / Embedding layers are torch library code in the reference and here; `components_ms` shows where the step's time
goes and `roofline` rates the GRU forward kernel, the longest of the step, against the FP32-pipe peak.  cpu_baseline / --impl reference = oracle/grusage_oracle.py (the composition pinned
against the reference's own classes) on all host threads, on a bounded sample of the same batch.
"""
from __future__ import annotations

import json
import os
import sys
import time

import torch
import torch.distributed as dist

METRIC = "grusage_train_graphs_per_sec"
T_FRAMES, F_DYN, MAP_S = 16, 6, 2048
POS_WEIGHT, LR, WD = 1.0, 1e-3, 5e-5
MODEL_KW = dict(dynamic_features_num=F_DYN, frames_num=T_FRAMES, gru_hidden_size=96, gru_num_layers=1, fc1dims=[96],
                sage_hidden_dims=[96, 96], fc2dims=[32], out_dim=1, num_st_types=256, emb_dim=8, dropout=0.25, negative_slope=0.1,
                global_pooling="double", mapenc_lane_embdim=8, mapenc_sage_hdims=[32, 32], map_attention_topk=5)
EXTENT = 2000.0


def make_map(seed=0):
    g = torch.Generator().manual_seed(1000 + seed)
    e = 4 * MAP_S
    return dict(float_features=torch.randn(MAP_S, 6, generator=g), bool_features=torch.rand(MAP_S, 3, generator=g) > 0.5,
                lane_type_cats=torch.randint(0, 6, (MAP_S,), generator=g),
                mgraph_edge_indexes=torch.stack([torch.randint(0, MAP_S, (e,), generator=g), torch.randint(0, MAP_S, (e,), generator=g)]),
                mseg_centroids=torch.rand(MAP_S, 2, generator=g) * EXTENT)


def make_batch(graphs, seed):
    from workloads import unit_map_graphs
    ei, bv, N = unit_map_graphs(graphs, seed=seed)
    g = torch.Generator().manual_seed(seed)
    return dict(x=torch.randn(N, T_FRAMES, F_DYN, generator=g), edge_index=ei, xsttype=torch.randint(0, 256, (N,), generator=g),
                xdims=torch.randn(N, 2, generator=g), pos_raw=torch.rand(N, T_FRAMES, 2, generator=g) * EXTENT, batch=bv,
                y=(torch.rand(graphs, 1, generator=g) > 0.5).float()), N, ei.size(1)


class Bag:
    def __init__(self, d, num_graphs):
        self.__dict__.update(d)
        self.num_graphs = num_graphs
        self.edge_attr = None


def _emit(line):
    """The JSON line goes to the real stdout that bench.py set aside (fd 1 itself is pointed at stderr there)."""
    main_mod = sys.modules.get("__main__")
    if hasattr(main_mod, "emit"):
        main_mod.emit(line)
    else:
        print(json.dumps(line), flush=True)


def env_rank():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def run_cpu(graphs_total, sample_graphs, steps, warmup, min_seconds):
    from oracle.grusage_oracle import GruSageOracle
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    model = GruSageOracle(**MODEL_KW, map_tensors=make_map())
    opt = torch.optim.Adam(model.parameters(), lr=LR, weight_decay=WD)
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(POS_WEIGHT))
    d, N, E = make_batch(sample_graphs, 0)
    data = Bag(d, sample_graphs)

    def step():
        opt.zero_grad()
        loss = crit(model(data), data.y)
        loss.backward()
        opt.step()
        return loss.item()

    for _ in range(warmup):
        step()
    t0, done = time.perf_counter(), 0
    while done < steps or (time.perf_counter() - t0) < min_seconds:
        step()
        done += 1
    dt = (time.perf_counter() - t0) / done
    return dict(graphs_per_s=sample_graphs / dt, ms=dt * 1e3, cores=cores, iters=done,
                sample=f"{sample_graphs} of {graphs_total} sequences of one batch ({N} nodes, {E} edges), full training step, "
                       f"{done} timed iterations after {warmup} warm-up")


def config(graphs, N=None, E=None):
    c = {"workload": "c2", "model": "GruSage, reference defaults (hidden 96, SageBlock [128,96,96], map 2048 segments / hidden 32, top-5, dropout 0.25)",
         "frames": T_FRAMES, "dynamic_features": F_DYN, "graphs_per_gpu": graphs, "optimizer": "Adam lr 1e-3 wd 5e-5",
         "loss": "BCEWithLogits(pos_weight)", "step": "zero_grad + forward + loss + backward (+ grad all-reduce at N>1) + Adam + loss.item()",
         "l2": "two batches alternate; activations of a batch exceed the 126 MB L2 at the default size",
         "parallelism": "graph-sharded data parallel, one flat-bucket NCCL all-reduce"}
    if N is not None:
        c.update(nodes_per_gpu=N, edges_per_gpu=E)
    return c


def main_reference(args):
    rank, _, _ = env_rank()
    if rank != 0:
        return
    r = run_cpu(args.c2_graphs, min(args.c2_graphs, 32), max(1, args.steps), max(1, args.warmup), 0.0)
    _emit({
        "impl": "reference", "metric": METRIC, "value": r["graphs_per_s"], "unit": "graphs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": r["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": config(args.c2_graphs),
        "cpu_baseline": {"value": r["graphs_per_s"], "unit": "graphs/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["graphs_per_s"], "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle/grusage_oracle.py: composition pinned bit-for-bit against the reference's own GruSage classes (tests/golden/grusage)"})


def main_ours(args):
    from bench import ClockSampler                     # same clocks / throttle sampling as the headline bench
    rank, local_rank, world = env_rank()
    assert torch.cuda.is_available(), "bench_c2.py needs a GPU (the product has no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import sldm_gnn_b200 as sg
    from sldm_gnn_b200 import _lib

    G = args.c2_graphs
    torch.manual_seed(0)
    model = sg.GruSage(**MODEL_KW, map_tensors=make_map()).to(dev)
    params = [p for p in model.parameters() if p.requires_grad]
    if world > 1:
        flat = torch.cat([p.detach().reshape(-1) for p in params])
        dist.broadcast(flat, src=0)
        off = 0
        with torch.no_grad():
            for p in params:
                p.copy_(flat[off:off + p.numel()].view_as(p)); off += p.numel()
    opt = torch.optim.Adam(params, lr=LR, weight_decay=WD)
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(POS_WEIGHT, device=dev))
    batches = []
    for j in range(2):
        d, N, E = make_batch(G, rank * 2 + j)
        host = {k: v.pin_memory() for k, v in d.items()}
        batches.append(dict(host=host, dev=Bag({k: v.to(dev) for k, v in host.items()}, G), N=N, E=E))
    N, E = batches[0]["N"], batches[0]["E"]
    h2d_bytes = sum(v.numel() * v.element_size() for v in batches[0]["host"].values())

    def step(data):
        opt.zero_grad(set_to_none=False) if world > 1 else opt.zero_grad()
        loss = crit(model(data), data.y)
        loss.backward()
        if world > 1:                               # one flat bucket, one all-reduce (mean over ranks: equal graph counts)
            bucket = torch.cat([p.grad.reshape(-1) for p in params])
            dist.all_reduce(bucket)
            bucket /= world
            off = 0
            for p in params:
                p.grad.copy_(bucket[off:off + p.numel()].view_as(p)); off += p.numel()
        opt.step()
        return loss.item()                          # the reference reads the loss every step (src/utils.py:226)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)
    for i in range(max(3, args.warmup)):
        step(batches[i % 2]["dev"])
    barrier()
    launches0 = _lib.lib.sldm_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_begin()
    t0.record()
    for i in range(args.steps):
        loss = step(batches[i % 2]["dev"])
    t1.record()
    barrier()
    sampler.mark_end()
    launches = _lib.lib.sldm_launch_count() - launches0
    ms_total = t0.elapsed_time(t1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:        # the step's loss and the parameters its Adam step left behind
        from bench import dump_outputs
        dump_outputs(args.dump_outputs, {"loss": torch.tensor([loss], dtype=torch.float64),
                                         **{"param." + k: p for k, p in model.named_parameters()}})

    # ---- end to end: the batch is copied from pinned host memory every step (prefetched one step ahead on a copy stream) ----
    copy_stream, main_stream = torch.cuda.Stream(device=dev), torch.cuda.current_stream(dev)

    def prefetch(i):
        with torch.cuda.stream(copy_stream):
            d = {k: v.to(dev, non_blocking=True) for k, v in batches[i % 2]["host"].items()}
            ev = torch.cuda.Event(); ev.record(copy_stream)
        return d, ev

    def consume(item):
        d, ev = item
        main_stream.wait_event(ev)
        for v in d.values():
            v.record_stream(main_stream)
        return step(Bag(d, G))

    e2e_steps = max(2, min(args.steps, 10))
    nxt = prefetch(0)
    for i in range(2):
        cur, nxt = nxt, prefetch(i + 1)
        consume(cur)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(e2e_steps):
        cur, nxt = nxt, prefetch(i + 3)
        consume(cur)
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)

    # ---- the same training step with forward and backward as captured CUDA graphs (GraphedGruSage): what the
    #      reference's real batch sizes (32 / 64 graphs) gain once the ~200 launches of a step are two graph launches ----
    # (captured before the component timings below: torch.cuda.make_graphed_callables must not find a live autograd
    #  graph of an earlier eager step -- its AccumulateGrad nodes belong to the default stream and a backward capture
    #  that has to synchronise with them is invalidated)
    graphed = None
    if world == 1 and G <= 256:
        try:
            import gc
            from sldm_gnn_b200.grusage import GraphedGruSage
            del cur, nxt
            gc.collect()
            gm = GraphedGruSage(model, max_nodes=max(b["N"] for b in batches) + 1, max_edges=max(b["E"] for b in batches),
                                max_graphs=G + 1, training=True)

            def gstep(data):
                opt.zero_grad()
                loss = crit(gm(data), data.y)
                loss.backward()
                opt.step()
                return loss.item()

            for i in range(5):
                gstep(batches[i % 2]["dev"])
            torch.cuda.synchronize()
            gsteps = max(args.steps, 50)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(gsteps):
                gstep(batches[i % 2]["dev"])
            b.record(); torch.cuda.synchronize()
            gms = a.elapsed_time(b) / gsteps
            graphed = {"ms_per_step": round(gms, 4), "graphs_per_sec": G / (gms * 1e-3), "steps": gsteps,
                       "what": "GraphedGruSage: padded static buffers, forward graph + backward graph behind autograd; loss, "
                               "Adam and loss.item() stay eager"}
            # ... and the whole step as ONE graph (GraphedTrainStep: zero_grad + forward + loss + backward + Adam)
            import torch.nn.functional as Fn
            from sldm_gnn_b200.grusage import GraphedTrainStep
            del gm
            gc.collect()
            pw = torch.tensor(POS_WEIGHT, device=dev)
            opt2 = torch.optim.Adam(params, lr=LR, weight_decay=WD, capturable=True, fused=True)
            ts = GraphedTrainStep(model, opt2, lambda lg, y, w: Fn.binary_cross_entropy_with_logits(lg, y, weight=w, pos_weight=pw, reduction="sum"),
                                  max_nodes=max(b["N"] for b in batches) + 1, max_edges=max(b["E"] for b in batches), max_graphs=G + 1)
            for i in range(5):
                ts(batches[i % 2]["dev"], batches[i % 2]["dev"].y).item()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0 = time.perf_counter()
            a.record()
            for i in range(gsteps):
                lossv = ts(batches[i % 2]["dev"], batches[i % 2]["dev"].y).item()
            b.record(); torch.cuda.synchronize()
            tms = a.elapsed_time(b) / gsteps
            graphed["one_graph_step"] = {"ms_per_step": round(tms, 4), "graphs_per_sec": G / (tms * 1e-3), "steps": gsteps, "last_loss": lossv,
                                         "what": "GraphedTrainStep: zero_grad + forward + BCE + backward + fused Adam in ONE graph; "
                                                 "per step: copy-in of the batch, one graph launch, loss.item()"}
        except Exception as exc:                   # must never take the headline line down
            import traceback
            graphed = {"error": repr(exc)[:300], "where": [l.strip() for l in traceback.format_exc().splitlines() if l.strip().startswith("File")][-8:]}

    # ---- where the time goes: forward stages with CUDA events (untimed for the headline), backward and optimizer as wholes ----
    comp = {}
    if rank == 0:
        data = batches[0]["dev"]

        def timed(fn, reps=5):
            fn(); torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                out = fn()
            b.record(); torch.cuda.synchronize()
            return a.elapsed_time(b) / reps, out

        comp["gru_last_hidden_fwd_training"], _ = timed(lambda: model._last_hidden(data.x))   # saves the gates for backward
        with torch.no_grad():
            comp["gru_fc1_embedding_fwd"], x1 = timed(lambda: _front(model, data))
            comp["map_encoder_sageblock_fwd"], emb = timed(lambda: model.map_encoder())
            comp["map_attention_fwd"], ctxv = timed(lambda: model.map_attention(data.pos_raw[:, -1, :], emb))
            xin = torch.cat([x1, ctxv], 1)
            comp["vehicle_sageblock_fwd"], xs = timed(lambda: model.sage(xin, data.edge_index))
            comp["readout_fwd"], _ = timed(lambda: model.global_pool(xs, data.batch, G))
        opt.zero_grad()
        comp["forward_total"], loss = timed(lambda: crit(model(data), data.y), reps=1)
        comp["backward_total"], _ = timed(lambda: torch.autograd.grad(crit(model(data), data.y), params), reps=1)
        comp["backward_total"] -= comp["forward_total"]
        comp = {k: round(v, 4) for k, v in comp.items()}

    times = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = times.tolist()
    if rank == 0:
        ms = ms_total / args.steps
        ms2 = ms_e2e / e2e_steps
        line = {"metric": METRIC, "value": G * world / (ms * 1e-3), "unit": "graphs/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": config(G, N, E),
                "clocks": clocks,
                "e2e": {"value": G * world / (ms2 * 1e-3), "unit": "graphs/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                        "ms_per_step": ms2, "steps": e2e_steps},
                "gpu_launches": int(launches), "components_ms": comp,
                "roofline": gru_roofline(N, comp.get("gru_last_hidden_fwd_training"), clocks)}
        if graphed is not None:
            line["cuda_graph"] = graphed
        if not args.no_cpu:
            r = run_cpu(G, min(G, 32), 1, 1, 10.0)
            line["cpu_baseline"] = {"value": r["graphs_per_s"], "unit": "graphs/s", "cores": r["cores"], "kind": "port",
                                    "sample": r["sample"], "ms_per_step": r["ms"]}
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


def gru_roofline(N, ms, clocks):
    """The step's dominant kernel is k_gru_fwd / k_gru_bwd (csrc/gru.cu): FP32 FMA work, bound by the FP32 pipe
    (128 FMA lanes per SM and clock), not by HBM or the tensor pipe -- reported against that peak at the SM clock
    sampled during the run."""
    import ctypes
    from sldm_gnn_b200 import _lib
    if not ms or os.environ.get("SLDM_DISABLE_FUSED_GRU", "0") == "1":
        return None
    sms = ctypes.c_int(0)
    _lib.check(_lib.lib.sldm_device_sm_count(ctypes.byref(sms)))
    mhz = float((clocks or {}).get("sm_mhz") or 0.0) or 1965.0
    hid = MODEL_KW["gru_hidden_size"]
    flops = 2.0 * N * T_FRAMES * 3 * hid * (hid + F_DYN)
    peak = sms.value * 128 * 2 * mhz * 1e6 / 1e12
    ach = flops / (ms * 1e-3) / 1e12
    return {"bound": "fp32_pipe", "kernel": "gru_last_hidden_fwd", "cuda_kernel": f"k_gru_fwd<{hid}, true>",
            "achieved": round(ach, 2), "peak": round(peak, 2), "unit": "TFLOP/s", "frac": round(ach / peak, 4),
            "traffic": None, "ms_per_launch": ms, "algorithmic_flops_per_launch": flops,
            "peak_source": f"{sms.value} SMs x 128 FMA/clk x 2 x {mhz:.0f} MHz (SM clock sampled during the run)",
            "note": "recurrent GEMM h.W_hh^T + gates, all T steps in one launch; SIMT FP32 (parity bar 1e-5 rules out "
                    "plain TF32; a 3xTF32 tcgen05 version is the next step)"}


def _front(model, data):
    h = model._last_hidden(data.x)
    x = torch.cat([h, data.xdims, model.st_emb(data.xsttype)], dim=1)
    for fc in model.fc1s:
        x = fc(x)
    return x


def main(args):
    if args.impl == "reference":
        main_reference(args)
    else:
        main_ours(args)
