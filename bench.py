#!/usr/bin/env python
"""bench.py -- SageBlock fwd+bwd throughput (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload batch|c4|c1|infer|c2] [--impl ours|reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one training pass of the hot path over one batch: CSR build from a fresh
edge_index, SageBlock forward, backward (dx and all parameter gradients) and -- at
N > 1 -- the single flat-bucket NCCL all-reduce of the gradients.

Workloads (SURVEY 8d; all synthetic, seeded, random-init weights):
  batch (default) : one mega-batch of 4096 unit map graphs per GPU (~0.82 M nodes,
                    ~4.1 M edges, block diagonal), SageBlock([128,128,128]); BASELINE
                    configs[2]/[4] shape.  Shards over ranks by whole graphs: weak scaling.
  c4              : one skewed graph, 1 M nodes / 10 M edges, SageBlock([128,128]): HBM
                    roofline stress (BASELINE configs[3]); replicas only at N > 1.
  c1              : 32 unit map graphs, SageBlock([64,64,64]) (BASELINE configs[0]).
  infer           : the batch shape, forward only under inference_mode (BASELINE configs[2]).
  c2              : BASELINE configs[1], the reference's FULL training step (GruSage + BCE + Adam) on our kernels; its own
                    metric (graphs/s) and file (bench_c2.py).  It is not the default because BASELINE's metric is quoted on
                    SageBlock fwd+bwd (edges/s, % of HBM roofline) and 80 % of that step is the GRU sequence head (our fused
                    FP32 kernels, csrc/gru.cu; profiles/r01m_bench_c2_1024.json): the SageBlock edge rate cannot be read off it.
value   = edge-layer traversals per second (E*L per step), whole job, inputs resident in HBM.
e2e     = the same through the public module call with pinned HOST inputs: H2D of x and
          edge_index, fwd+bwd, D2H of the loss, all inside the timed region.
roofline= the dominant kernel (longest share of the step), algorithmic bytes / its own
          CUDA-event time / measured HBM peak; roofline_step = SURVEY 8d's per-layer
          fwd+bwd byte model for the whole step.
--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<name>.npy (float32; rank 0's
          share at N > 1), so that two builds run with the same arguments can be compared output for output:
          out = block output, dx = gradient of x, grad.<parameter> = every parameter gradient (no dx / grad.* for
          infer).  Of out and dx only a fixed, seeded sample of DUMP_ROWS rows is written (all rows of a smaller
          output), at most 32 MB in all at width 128.  c2 writes the loss and every parameter after the Adam step.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# stdout carries ONE JSON line and nothing else.  NCCL prints its version banner with printf at communicator init
# (NCCL_DEBUG_FILE does not catch it), so the real stdout is kept aside and file descriptor 1 is pointed at stderr for
# everything else -- this process's own prints and any library's.
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
if __name__ == "__main__":
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
else:
    _JSON_OUT = sys.stdout


def emit(line: dict) -> None:
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

WORKLOADS = {
    "batch": dict(kind="graphs", graphs=4096, hdims=[128, 128, 128], cpu_sample_graphs=4096),
    "c1": dict(kind="graphs", graphs=32, hdims=[64, 64, 64], cpu_sample_graphs=32),
    "c4": dict(kind="skewed", nodes=1_000_000, edges=10_000_000, hdims=[128, 128], cpu_sample_graphs=None),
    # BASELINE configs[2]: batched inference, hidden 128 -- one mega-batch of 4096 graphs, forward only (inference_mode)
    "infer": dict(kind="graphs", graphs=4096, hdims=[128, 128, 128], cpu_sample_graphs=4096, forward_only=True),
}
SLOPE = 0.1
METRIC = "sageblock_fwd_bwd_edges_per_sec"     # --workload infer reports forward-only traversals under the same name, flagged in config.step
DUMP_ROWS = 32768


def dump_rows(n):
    """Row indices of the --dump-outputs sample of an [n, F] output: all rows when n <= DUMP_ROWS, else the same
    seeded DUMP_ROWS rows (ascending) for every build and run."""
    if n <= DUMP_ROWS:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values


def dump_outputs(dirname, arrays):
    """--dump-outputs: each tensor as dirname/<name>.npy, float64 kept, every other dtype as float32."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        np.save(os.path.join(dirname, name + ".npy"), t.numpy() if t.dtype == torch.float64 else t.float().numpy())


def env_rank():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_inputs(wl, seed):
    from workloads import unit_map_graphs, skewed_graph
    g = torch.Generator().manual_seed(1000 + seed)
    if wl["kind"] == "graphs":
        ei, bv, N = unit_map_graphs(wl["graphs"], seed=seed)
        graphs = wl["graphs"]
    else:
        N = wl["nodes"]
        ei = skewed_graph(N, wl["edges"], seed=seed)
        graphs, bv = 1, None
    x = torch.randn(N, wl["hdims"][0], generator=g)
    return x, ei, N, graphs, bv


# CUDA kernel behind each timed group, and how many times it runs per layer and step (fwd+bwd)
KERNEL_NAMES = {"segment_mean_fwd": "k_segment_rows_lean", "project_ln_act_fwd": "k_sage_tc<NT, MODE_FWD>",
                "segment_sum_bwd": "k_segment_rows_lean (transpose CSR)", "ln_bwd": "k_ln_bwd_rows",
                "dgrad": "k_split_weights_t + k_sage_tc<NT, MODE_DGRAD>", "wgrad": "k_wgrad_tc<NB> + k_reduce_parts x2",
                "csr_build": "k_convert + k_digit_hist + k_onesweep_pass x3 + k_rowptr_from_sorted",
                "layer_backward": "k_ln_bwd_rows + k_sage_tc<NT, MODE_DGRAD> + k_wgrad_tc + k_reduce_parts + k_segment_rows_lean",
                "readout_mean_max_fwd": "membership CSR build + k_readout_fwd", "readout_bwd": "k_readout_bwd_graph",
                "map_attention_fwd": "k_map_attention_fwd", "map_attention_bwd": "k_map_attention_bwd + membership CSR + k_map_attention_demb",
                "collate_32_graphs": "k_concat_chunks x5 + k_collate_edge_index + k_batch_from_ptr (+ host table upload)"}
# every group that is ONE dominant kernel (the candidates of `roofline`), launches per layer and step
KERNEL_LAUNCHES_PER_LAYER = {"segment_mean_fwd": 1, "project_ln_act_fwd": 1, "ln_bwd": 1, "dgrad": 1, "wgrad": 1,
                             "segment_sum_bwd": 1}


def committed_ncu_traffic(workload, group):
    """DRAM bytes per launch from the latest committed ncu --set full capture (profiles/*_traffic.json), or None.
    Reported beside the roofline as `traffic_ncu_committed`: it is NOT a measurement of this run (`traffic` is null)."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    path = files[-1] if files else ""
    if group is None or not os.path.exists(path):
        return None
    try:
        v = json.load(open(path)).get(workload, {}).get(group)
        return None if v is None else {"bytes_per_launch": v, "source": os.path.relpath(path, ROOT)}
    except Exception:
        return None


# ------------------------------------------------------------------ byte models --
def layer_bytes_fwd_bwd(N, E, Fin, Fout, s=4):
    """SURVEY 8d: 2E(Fin s + 4) + N s (6 Fin + 5 Fout) + 28 N per layer, fwd+bwd (training)."""
    return 2 * E * (Fin * s + 4) + N * s * (6 * Fin + 5 * Fout) + 28 * N


def layer_bytes_fwd_bwd_cache_perfect(N, E, Fin, Fout, s=4):
    """8d's own lower bound: the two gathers read every row once (E*Fin*s -> N*Fin*s), indices still cost 4 B per edge."""
    return 2 * (4 * E + N * Fin * s) + N * s * (6 * Fin + 5 * Fout) + 28 * N


def layer_bytes_fwd_bwd_bf16feat(N, E, Fin, Fout):
    """bf16 FEATURE storage (x, agg, out in 2 bytes; xhat, every gradient and all accumulation in fp32), the tensors
    the kernels actually move, per layer fwd+bwd: forward gather E(2Fin+4) + 4(N+1) + agg write 2N Fin; projection
    reads agg, x (2 x 2N Fin), writes out (2N Fout) + xhat (4N Fout) + rstd; backward as fp32 (8d) except that the
    weight gradient reads the bf16 agg / x."""
    fwd = E * (2 * Fin + 4) + 4 * (N + 1) + 2 * N * Fin + N * (4 * Fin + 2 * Fout + 4 * Fout) + 4 * N
    bwd = N * 4 * (3 * Fout) + N * 4 * (Fout + 2 * Fin) + N * (4 * Fout + 4 * Fin) + E * (Fin * 4 + 4) + 4 * (N + 1) + 3 * N * Fin * 4 + 12 * N
    return fwd + bwd


def csr_bytes(N, E):
    return 16 * E + 8 * E + 8 * (N + 1)


def bind_to_gpu_numa_node(index):
    """Pin this rank's host threads to the CPUs NVML reports as local to its GPU, BEFORE the pinned staging buffers are
    allocated (first touch places them on that NUMA node): with 8 ranks feeding 486 MB per step each, host memory that
    sits across the socket link halves the H2D rate.  Best effort: returns the CPU count bound, or None."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = [i for i in range(ncpu) if (int(words[i // 64]) >> (i % 64)) & 1]
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            return len(allowed)
    except Exception:
        pass
    return None


# ---------------------------------------------------------------- clock sampler --
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t_begin = self.t_end = None

    def mark_begin(self):
        self.t_begin = time.time()

    def mark_end(self):
        self.t_end = time.time()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.index), "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [r for (t, r) in self.rows if self.t_begin is not None and self.t_begin <= t <= (self.t_end or t) + 0.05]
        window = "timed region"
        if len(inside) < 3:   # region shorter than a few sampling periods: use everything since warm-up started
            inside, window = [r for (_, r) in self.rows], "warm-up + timed region (timed region < 3 samples)"
        for r in inside:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


# ------------------------------------------------------------------- CPU legs --
def upstream_gradient(N, width):
    """dL/dout of the step, the same tensor in both arms: stands in for whatever follows the block."""
    return torch.randn(N, width, generator=torch.Generator().manual_seed(7 + N))


def cpu_reference_step(block, x, ei, w, forward_only=False):
    if forward_only:
        with torch.inference_mode():
            block(x, ei)
        return
    xr = x.clone().requires_grad_(True)
    y = block(xr, ei)
    y.backward(w)
    block.zero_grad(set_to_none=True)


def cpu_sample(wl, seed=0):
    """The workload of the CPU legs: the WHOLE batch for the graph workloads (seed 0, the GPU arm's first batch);
    a 1/10-scale graph for c4 (the full one is ~4 s per step and tens of GB of [E, F] intermediates)."""
    from workloads import skewed_graph
    if wl["kind"] == "graphs":
        x, ei, N, graphs, _ = make_inputs(wl, seed)
        desc = f"the full batch: {graphs} unit map graphs, {N} nodes, {ei.size(1)} edges"
    else:
        N, E = wl["nodes"] // 10, wl["edges"] // 10
        ei = skewed_graph(N, E, seed=seed)
        x = torch.randn(N, wl["hdims"][0], generator=torch.Generator().manual_seed(1000 + seed))
        desc = f"1/10-scale skewed graph ({N} nodes, {E} edges) -- NOT the full configuration"
        graphs = 1
    return x, ei, N, graphs, desc


def run_cpu(wl, steps, warmup, min_seconds=0.0, max_seconds=1e9):
    """The reference's CPU path: oracle/sage_oracle.py restates PyG 2.7.0 SAGEConv with the same ATen
    CPU operators (torch-geometric is not installable here), all host threads."""
    from oracle.sage_oracle import SageBlockOracle
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    blk = SageBlockOracle(wl["hdims"], dropout=None, negative_slope=SLOPE)
    x, ei, N, graphs, desc = cpu_sample(wl)
    w = upstream_gradient(N, wl["hdims"][-1])
    fo = bool(wl.get("forward_only"))
    for _ in range(warmup):
        cpu_reference_step(blk, x, ei, w, fo)
    t0 = time.perf_counter()
    done = 0
    while (done < steps or (time.perf_counter() - t0) < min_seconds) and (done == 0 or (time.perf_counter() - t0) < max_seconds):
        cpu_reference_step(blk, x, ei, w, fo)
        done += 1
    steps = done
    dt = (time.perf_counter() - t0) / steps
    L = len(wl["hdims"]) - 1
    return dict(edges_per_s=ei.size(1) * L / dt, graphs_per_s=graphs / dt, ms=dt * 1e3, cores=cores,
                sample=desc + (", forward only" if fo else ", fwd+bwd from the fixed upstream gradient"), iters=steps,
                N=N, E=ei.size(1), graphs=graphs)


def main_reference(args, wl):
    """--impl reference: the reference's CPU implementation of the path (the oracle port; PyG is not installable
    here) on all host cores, the same workload, loss and config keys as the GPU arm.  Rank 0 only."""
    rank, _, world = env_rank()
    if rank != 0:
        return
    r = run_cpu(wl, max(1, args.steps), max(1, args.warmup), max_seconds=240.0)
    full = wl["kind"] == "graphs"
    cfg = workload_config(args.workload, wl, r["N"] if full else wl["nodes"], r["E"] if full else wl["edges"], r["graphs"])
    line = {
        "impl": "reference", "metric": METRIC, "value": r["edges_per_s"], "unit": "edges/s", "n_gpus": args.gpus,
        "steps": r["iters"], "warmup": max(1, args.warmup), "ms_per_step": r["ms"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "graphs_per_sec": r["graphs_per_s"],
        "cpu_baseline": {"value": r["edges_per_s"], "unit": "edges/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["edges_per_s"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle/sage_oracle.py (torch CPU restatement of PyG 2.7.0 SAGEConv; torch-geometric is not installable offline); "
                "one process, all host cores, whatever --gpus says",
    }
    emit(line)


def workload_config(name, wl, N, E, graphs):
    c = {"workload": name, "hdims": wl["hdims"], "negative_slope": SLOPE, "dropout": None,
         "step": ("csr_build + forward under inference_mode (no backward)" if wl.get("forward_only") else
                  "csr_build + forward + backward from a fixed upstream gradient dL/dout (+ grad all-reduce at N>1)"),
         "l2": "inputs and saved tensors exceed the 126 MB L2 (x alone is N*F*4 B); two input batches alternate"}
    if N is not None:
        c.update(nodes_per_gpu=N, edges_per_gpu=E, graphs_per_gpu=graphs)
    c["parallelism"] = "graph-sharded data parallel, per-layer gradient buckets all-reduced (NCCL) under the rest of backward" if name != "c4" else "replicas only"
    return c


# -------------------------------------------------------------------- GPU leg --
def widened_groups(sg, x, out, batch_vec, num_graphs, N, s):
    """Timing groups of the components either side of the block (SURVEY 8f): readout, mini-batch assembly, map attention."""
    groups = {}
    # graph readout on the block's output (SURVEY 8f-1): membership CSR + fused mean|max forward, and its backward
    G = int(num_graphs)
    bv = batch_vec.to(x.device)
    Fo = out.size(1)
    xo = out.detach().clone().requires_grad_(True)
    ro = sg.global_mean_max_pool(xo, bv, G)
    dro = torch.randn_like(ro)
    groups["readout_mean_max_fwd"] = (lambda: sg.global_mean_max_pool(out, bv, G), N * Fo * s + G * 2 * Fo * s + 8 * N)
    groups["readout_bwd"] = (lambda: torch.autograd.grad(ro, xo, dro, retain_graph=True), N * Fo * s + N * Fo * s + 4 * N)   # x from HBM once (its second sweep hits L2), dx written
    # mini-batch assembly (SURVEY 8f-2) at the reference's DataLoader batch size: 32 device-resident unit graphs with the
    # fields of a pack (x [n,T,6], edge_index, xsttype, xdims, pos_raw, y); timed end to end (host tables + kernels)
    from workloads import unit_map_graphs
    items, nb = [], 0
    for gidx in range(32):
        eg, _, ng = unit_map_graphs(1, seed=100 + gidx)
        d = dict(x=torch.randn(ng, 16, 6), edge_index=eg, xsttype=torch.randint(0, 5, (ng,)), xdims=torch.randn(ng, 2),
                 pos_raw=torch.randn(ng, 16, 2), y=torch.zeros(1, 4))
        nb += 2 * sum(v.numel() * v.element_size() for v in d.values()) + 8 * ng
        items.append(sg.GraphData(**{k: v.to(x.device) for k, v in d.items()}))
    groups["collate_32_graphs"] = (lambda: sg.collate(items), nb)
    # map attention (SURVEY 8f-3): one position per node of the batch, a 2048-segment map, 32-d map embeddings, K = 5
    Sm, Dm = 2048, 32
    gm = torch.Generator().manual_seed(11)
    att = sg.MapSpatialAttention(torch.rand(Sm, 2, generator=gm) * 2000.0, 5).to(x.device)
    posm = (torch.rand(N, 2, generator=gm) * 2000.0).to(x.device)
    embm = torch.randn(Sm, Dm, generator=gm).to(x.device).requires_grad_(True)
    ctxm = att(posm, embm)
    dctxm = torch.randn_like(ctxm)
    groups["map_attention_fwd"] = (lambda: att(posm, embm.detach()), N * (8 + 5 * Dm * s + Dm * s + 5 * 16) + Sm * (8 + Dm * s))
    groups["map_attention_bwd"] = (lambda: torch.autograd.grad(ctxm, [embm] + list(att.parameters()), dctxm, retain_graph=True),
                                   N * (Dm * s + 5 * Dm * s + 5 * 16) + 2 * 5 * N * Dm * s // 2 + Sm * Dm * s)
    return groups


def time_kernels(blk, x, ei, N, E, hdims, peak_gbs, batch_vec=None, num_graphs=None, only=None):
    """Per-kernel-group CUDA-event timing of layer 0 (through the C-ABI, on torch's current stream)."""
    import sldm_gnn_b200 as sg
    from sldm_gnn_b200 import ops
    Fin, Fout = hdims[0], hdims[1]
    conv, ln = blk.convs[0], blk.posts[0][0]
    p = (conv.lin_l.weight, conv.lin_l.bias, conv.lin_r.weight, ln.weight, ln.bias)
    csr = sg.build_csr(ei, N)
    _, out, agg, xhat, rstd = ops.layer_forward(x, csr, *p, ln.eps, SLOPE, True)
    dout = torch.randn(out.shape, dtype=torch.float32, device=out.device)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=x.device)

    def timed(fn, reps=5):
        ts = []
        for _ in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); b.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return ts[len(ts) // 2]

    s = 4
    sf = 2 if x.dtype == torch.bfloat16 else 4      # bytes per stored FEATURE (x, agg, out); gradients / xhat stay fp32
    seg_fwd = (lambda: ops.segment_mean_bf16(x, csr)) if sf == 2 else (lambda: sg.segment_reduce(x, csr))
    from sldm_gnn_b200 import _lib as L_
    bb = ops.backward_buffers(N, Fin, Fout, E, x.device, True)
    bargs = (dout, x, agg, xhat, rstd, csr, p[0], p[2], p[3], p[4], SLOPE, True)
    ops.layer_backward(*bargs, bufs=bb)          # fills dz / dagg / dxroot / partials for the single-stage launches
    groups = {
        "csr_build": (lambda: sg.build_csr(ei, N), csr_bytes(N, E)),
        "segment_mean_fwd": (seg_fwd, E * (Fin * sf + 4) + 4 * (N + 1) + N * Fin * sf),
        "project_ln_act_fwd": (lambda: ops.project_forward(agg, x, *p, ln.eps, SLOPE, True),
                               N * (2 * Fin * sf + Fout * sf + Fout * s) + 4 * N),
        "layer_backward": (lambda: ops.layer_backward(dout, x, agg, xhat, rstd, csr, p[0], p[2], p[3], p[4], SLOPE, True),
                           N * (3 * Fout * s + 2 * Fin * sf + 2 * Fin * s) + 12 * N + E * (Fin * s + 4) + 4 * (N + 1)),
        # the kernels of layer_backward one at a time (include/sldm_sage.h SLDM_BWD_STAGE_*), on the buffers of a full call
        "ln_bwd": (lambda: ops.layer_backward(*bargs, stages=L_.BWD_STAGE_LN, bufs=bb), 3 * N * s * Fout + 4 * N),
        "dgrad": (lambda: ops.layer_backward(*bargs, stages=L_.BWD_STAGE_DGRAD, bufs=bb), N * s * (Fout + 2 * Fin) + 4 * N),
        "wgrad": (lambda: ops.layer_backward(*bargs, stages=L_.BWD_STAGE_WGRAD, bufs=bb), N * (s * Fout + 2 * Fin * sf)),
        "segment_sum_bwd": (lambda: ops.layer_backward(*bargs, stages=L_.BWD_STAGE_GATHER, bufs=bb),
                            E * (Fin * s + 4) + 4 * (N + 1) + 3 * N * Fin * s),
    }
    if batch_vec is not None:
        try:     # the widened components (SURVEY 8f) must never take the headline measurement down
            groups.update(widened_groups(sg, x, out if out.dtype == torch.float32 else out.float(), batch_vec, num_graphs, N, s))
        except Exception as exc:
            groups["widened_components"] = (lambda: (_ for _ in ()).throw(RuntimeError(repr(exc)[:200])), 0)
    res = {}
    core = ("csr_build", "segment_mean_fwd", "project_ln_act_fwd", "layer_backward", "ln_bwd", "dgrad", "wgrad", "segment_sum_bwd")
    for k, (fn, nbytes) in groups.items():
        if only is not None and k not in only:
            continue
        try:
            fn(); torch.cuda.synchronize()
            ms = timed(fn)
        except Exception as exc:             # the widened components must never take the headline measurement down
            if k in core:
                raise
            res[k] = {"error": repr(exc)[:200]}
            continue
        res[k] = {"ms": round(ms, 4), "algorithmic_bytes": nbytes, "gbs": round(nbytes / ms / 1e6, 1),
                  "frac_hbm": round(nbytes / ms / 1e6 / peak_gbs, 4)}
    return res


def c4_record(dev, peak_gbs, steps=10):
    """BASELINE configs[3] inside the default line (so the driver-run record carries the HBM-stress configuration):
    one skewed graph, 1 M nodes / 10 M edges, SageBlock([128,128]), CSR build + forward + backward."""
    import sldm_gnn_b200 as sg
    wl = WORKLOADS["c4"]
    hdims = wl["hdims"]
    x_h, ei_h, N, _, _ = make_inputs(wl, 0)
    E = ei_h.size(1)
    torch.manual_seed(0)
    blk = sg.SageBlock(hdims, dropout=None, negative_slope=SLOPE).to(dev)
    x = x_h.to(dev).requires_grad_(True)
    ei = ei_h.to(dev)
    w = upstream_gradient(N, hdims[-1]).to(dev)

    def step():
        blk.clear_cache()
        blk.zero_grad(set_to_none=True)
        x.grad = None
        blk(x, ei).backward(w)

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        step()
    t1.record()
    t1.synchronize()
    ms = t0.elapsed_time(t1) / steps
    nbytes = layer_bytes_fwd_bwd(N, E, hdims[0], hdims[1]) + csr_bytes(N, E)
    kern = time_kernels(blk, x.detach(), ei, N, E, hdims, peak_gbs,
                        only=("segment_mean_fwd", "project_ln_act_fwd", "dgrad", "wgrad", "segment_sum_bwd", "csr_build"))
    return {"workload": "c4", "nodes": N, "edges": E, "hdims": hdims, "steps": steps, "ms_per_step": ms,
            "edges_per_sec": E * (len(hdims) - 1) / (ms * 1e-3),
            "roofline_step_frac": nbytes / ms / 1e6 / peak_gbs, "algorithmic_bytes": nbytes,
            "gather_frac": kern["segment_mean_fwd"]["frac_hbm"], "kernels": kern,
            "note": "true random gather (no L2 absorption): SURVEY 8d's byte model is honest here"}


def cabi_host_record(blk, b, hdims, slope, N, E, fwd_only, calls=3):
    """The same step through the C-ABI entry points that take HOST buffers (include/sldm_sage.h:
    sldm_sage_block_forward_host / _train_host -- the call a host without torch would bind, INTEGRATION.md section 3):
    every call copies x and edge_index (and the upstream gradient) to the device, builds the CSR, runs the layers and
    copies the output (and dx and every parameter gradient) back, synchronously.  Pinned host buffers; wall clock
    around the blocking call.  It moves 2-4x the bytes of the module-level e2e (whose loss stays a 4-byte read)."""
    import ctypes as C
    from sldm_gnn_b200 import _lib
    L = len(hdims) - 1
    pin = lambda t: t.detach().to("cpu", torch.float32).contiguous().pin_memory()
    pbufs = []
    for l in range(L):
        pbufs += [pin(blk.convs[l].lin_l.weight), pin(blk.convs[l].lin_l.bias), pin(blk.convs[l].lin_r.weight),
                  pin(blk.posts[l][0].weight), pin(blk.posts[l][0].bias)]
    params = (C.c_void_p * len(pbufs))(*[t.data_ptr() for t in pbufs])
    hd = (C.c_int32 * (L + 1))(*hdims)
    x_h, ei_h = b["x_h"], b["ei_h"]
    out_h = torch.empty((N, hdims[-1]), dtype=torch.float32).pin_memory()
    h2d = x_h.numel() * 4 + ei_h.numel() * 8
    d2h = out_h.numel() * 4
    if fwd_only:
        call = lambda: _lib.check(_lib.lib.sldm_sage_block_forward_host(
            x_h.data_ptr(), ei_h.data_ptr(), N, E, hd, L, params, 1e-5, slope, out_h.data_ptr()))
    else:
        w_h = b["w"].detach().to("cpu", torch.float32).contiguous().pin_memory()
        dx_h = torch.empty_like(x_h).pin_memory()
        gbufs = [torch.empty_like(t).pin_memory() for t in pbufs]
        grads = (C.c_void_p * len(gbufs))(*[t.data_ptr() for t in gbufs])
        h2d += w_h.numel() * 4
        d2h += dx_h.numel() * 4 + sum(t.numel() * 4 for t in gbufs)
        call = lambda: _lib.check(_lib.lib.sldm_sage_block_train_host(
            x_h.data_ptr(), ei_h.data_ptr(), N, E, hd, L, params, 1e-5, slope, w_h.data_ptr(), out_h.data_ptr(),
            dx_h.data_ptr(), grads))
    call()                                          # warm-up: fills the library's device pool
    t0 = time.perf_counter()
    for _ in range(calls):
        call()
    ms = (time.perf_counter() - t0) * 1e3 / calls
    return {"entry": "sldm_sage_block_forward_host" if fwd_only else "sldm_sage_block_train_host", "ms_per_call": round(ms, 3),
            "value": E * L / (ms * 1e-3), "unit": "edges/s", "h2d_bytes_per_call": int(h2d), "d2h_bytes_per_call": int(d2h),
            "calls": calls, "note": "blocking C call, pinned host buffers in and out, no overlap between copies and kernels"}


def time_graphed(blk, batches, hdims, dev, fwd_only, steps=200):
    """ms per step of the small workload through GraphedSageBlock (one bucket sized for the batch): inference = copy-in
    + one graph launch + copy-out; training = forward graph + backward graph behind autograd.  Inputs alternate."""
    Nmax = max(b["N"] for b in batches) + 1
    Emax = max(b["E"] for b in batches)
    res = {"bucket": {"max_nodes": Nmax, "max_edges": Emax}}
    for mode in (("inference",) if fwd_only else ("inference", "training")):
        g = blk.graphed(Nmax, Emax, training=(mode == "training"))

        def step(b):
            if mode == "inference":
                return g(b["x"].detach(), b["ei"])
            blk.zero_grad(set_to_none=True)
            x = b["x"].detach().requires_grad_(True)
            g(x, b["ei"]).backward(b["w"])
            return x.grad

        for i in range(10):
            step(batches[i % 2])
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0 = time.perf_counter()
        t0.record()
        for i in range(steps):
            step(batches[i % 2])
        t1.record()
        host_ms = (time.perf_counter() - h0) * 1e3 / steps
        t1.synchronize()
        res[mode] = {"ms_per_step": t0.elapsed_time(t1) / steps, "host_enqueue_ms_per_step": round(host_ms, 4), "steps": steps}
    return res


def main_ours(args, wl):
    rank, local_rank, world = env_rank()
    assert torch.cuda.is_available(), "bench.py needs a GPU (the product has no CPU fallback)"
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import sldm_gnn_b200 as sg
    from sldm_gnn_b200 import _lib
    from sldm_gnn_b200.parallel import GraphDataParallel

    hdims = wl["hdims"]
    L = len(hdims) - 1
    bf16 = args.dtype == "bf16"
    if bf16 and not all(sg.ops.bf16_supported(hdims[l], hdims[l + 1]) for l in range(L)):
        raise SystemExit(f"--dtype bf16: hdims {hdims} are not covered by the bf16 kernels")
    torch.manual_seed(0)
    blk = sg.SageBlock(hdims, dropout=None, negative_slope=SLOPE).to(dev)
    ddp = GraphDataParallel(blk)
    # two independent batches per rank, alternated, so nothing is reused across steps
    batches = []
    for j in range(2):
        seed = (rank * 2 + j) if args.workload != "c4" else j
        x_h, ei_h, N, graphs, bv = make_inputs(wl, seed)
        if bf16:
            x_h = x_h.to(torch.bfloat16)           # the features are STORED as bf16: half the H2D bytes, half the HBM rows
        batches.append(dict(x_h=x_h.pin_memory(), ei_h=ei_h.pin_memory(), N=N, E=ei_h.size(1), graphs=graphs, bv=bv))
    for b in batches:
        b["x"] = b["x_h"].to(dev).requires_grad_(True)
        b["ei"] = b["ei_h"].to(dev)
        # fixed upstream gradient dL/dout: stands in for whatever follows the block (pooling, head, loss)
        b["w"] = upstream_gradient(b["N"], hdims[-1]).to(dev)
        if bf16:
            b["w"] = b["w"].to(torch.bfloat16)     # dL/dout has the dtype of the block's output
    N, E, graphs = batches[0]["N"], batches[0]["E"], batches[0]["graphs"]

    fwd_only = bool(wl.get("forward_only"))

    def step(b, x=None, ei=None):
        x = b["x"] if x is None else x
        ei = b["ei"] if ei is None else ei
        blk.clear_cache()                      # every batch is a new graph: CSR build is part of the step
        if fwd_only:                           # inference (test.py:136): no autograd graph, nothing saved
            with torch.inference_mode():
                return blk(x.detach(), ei)
        if world > 1:
            ddp.zero_grad()
            ddp.expect_sync(local_weight=b["graphs"])   # buckets leave for the all-reduce as backward finishes them
        else:
            blk.zero_grad(set_to_none=True)             # one GPU: the reference's own loop (optimizer.zero_grad(), src/utils.py:219)
        x.grad = None
        y = (ddp if world > 1 else blk)(x, ei)
        y.backward(b["w"])
        if world > 1:
            ddp.sync_gradients(local_weight=b["graphs"])
        return y.detach()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    overlap_check = None
    if world > 1 and not fwd_only:
        # The overlapped exchange (buckets written by the kernels and all-reduced from inside backward) must give the
        # SAME bits as the plain one (autograd accumulation, everything exchanged after backward) on the same batch.
        def grads_of(b, overlap):
            ddp.zero_grad()
            b["x"].grad = None
            if overlap:
                ddp.expect_sync(local_weight=b["graphs"])
            blk.clear_cache()
            ddp(b["x"], b["ei"]).backward(b["w"])
            ddp.sync_gradients(local_weight=b["graphs"])
            return ddp.flat_grad.clone()

        for _ in range(3):
            ga, gb = grads_of(batches[0], True), grads_of(batches[0], False)
            same = torch.equal(ga, gb)
            flag = torch.tensor([0 if same else 1], device=dev)
            dist.all_reduce(flag)
            overlap_check = "ok" if int(flag) == 0 else "MISMATCH"
            assert overlap_check == "ok", "overlapped gradient exchange differs from the plain exchange"

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.5)                        # let nvidia-smi come up before the load starts
    # settle: a fresh box pages the CUDA libraries in and ramps clocks during the first few hundred ms of work (a
    # 10-step run measured 6.1 ms/step cold against 4.5 warm).  The per-kernel-group timing runs first on every rank
    # (~0.5 s of the same kernels, untimed for the headline), then the W warm-up steps, then the K timed steps.
    peak_gbs, peak_src = measured_peaks()
    kern = None if args.skip_kernel_timing else time_kernels(blk, batches[0]["x"].detach(), batches[0]["ei"], N, E, hdims, peak_gbs, batches[0]["bv"], batches[0]["graphs"])
    # every step's output is held until the next one returns (the timed loop keeps the last for --dump-outputs), so the
    # warm-up holds it the same way: the timed steps then find both output blocks in the caching allocator
    for i in range(max(3, args.warmup)):
        y = step(batches[i % 2])
    barrier()
    launches0 = _lib.lib.sldm_launch_count()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    sampler.mark_begin()
    t0.record()
    h0 = time.perf_counter()
    for i in range(args.steps):
        y = step(batches[i % 2])
    host_enqueue_ms = (time.perf_counter() - h0) * 1e3 / args.steps   # host time to ENQUEUE a step (no sync inside)
    t1.record()
    barrier()
    sampler.mark_end()
    launches = _lib.lib.sldm_launch_count() - launches0
    ms_total = t0.elapsed_time(t1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:        # before the e2e steps below overwrite the gradients
        rows = dump_rows(y.size(0)).to(dev)
        arrays = {"out": y.index_select(0, rows)}
        if not fwd_only:
            arrays["dx"] = batches[(args.steps - 1) % 2]["x"].grad.index_select(0, rows)
            arrays.update({"grad." + k: p.grad for k, p in blk.named_parameters()})
        dump_outputs(args.dump_outputs, arrays)
    del y

    # ---- end to end: pinned host inputs -> H2D -> step -> D2H of the step's metric, every step ----
    # Input pipeline as a training loop would run it: the H2D copy of step i+1 is issued on a copy stream while
    # step i computes (double-buffered device inputs); every step's copies and its D2H read are inside the timed region.
    e2e_steps = max(2, min(args.steps, 10))
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream(dev)

    def prefetch(i):
        b = batches[i % 2]
        with torch.cuda.stream(copy_stream):
            xd = b["x_h"].to(dev, non_blocking=True)
            eid = b["ei_h"].to(dev, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return b, xd, eid, ev

    out_h = torch.empty((N, hdims[-1]), dtype=torch.bfloat16 if bf16 else torch.float32).pin_memory() if fwd_only else None

    def consume(item):
        b, xd, eid, ev = item
        main_stream.wait_event(ev)
        xd.record_stream(main_stream); eid.record_stream(main_stream)
        y = step(b, xd if fwd_only else xd.requires_grad_(True), eid)
        if fwd_only:                      # inference: the result IS the [N, Fout] output -- it comes back to the host
            out_h[: y.size(0)].copy_(y[: out_h.size(0)], non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
            return float(out_h[0, 0])
        return y.sum().item()             # training: .item() = the D2H read of the step's metric

    nxt = prefetch(0)
    for i in range(2):
        cur, nxt = nxt, prefetch(i + 1)
        consume(cur)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(e2e_steps):
        cur, nxt = nxt, prefetch(i + 3)     # exactly one H2D (x + edge_index) is issued per timed step
        loss_host = consume(cur)
    main_stream.wait_event(nxt[3])          # the last copy issued inside the region must finish inside it
    e1.record()
    barrier()
    e2e_ms_total = e0.elapsed_time(e1)
    assert loss_host == loss_host

    # ---- the same step through captured CUDA graphs (GraphedSageBlock): what the launch-bound small workloads gain ----
    graphed = None
    if args.workload == "c1" and world == 1:
        try:
            graphed = time_graphed(blk, batches, hdims, dev, fwd_only)
        except Exception as exc:                  # must never take the headline line down
            graphed = {"error": repr(exc)[:300]}
    cabi = None
    if world == 1 and not bf16 and args.workload in ("batch", "infer", "c1"):
        try:
            cabi = cabi_host_record(blk, batches[0], hdims, SLOPE, N, E, fwd_only)
        except Exception as exc:                  # must never take the headline line down
            cabi = {"error": repr(exc)[:300]}
    grad_sync = None
    if world > 1 and not fwd_only:               # after the exchange every rank must hold the SAME gradients, bit for bit
        chk = ddp.flat_grad.double().sum().view(1)
        allc = [torch.zeros_like(chk) for _ in range(world)]
        dist.all_gather(allc, chk)
        grad_sync = "ok" if all(torch.equal(allc[0], c) for c in allc) and bool(torch.isfinite(chk).all()) else "MISMATCH"
        assert grad_sync == "ok", "gradient exchange left the ranks with different gradients"

    t = torch.tensor([ms_total, e2e_ms_total, float(E), float(graphs)], dtype=torch.float64, device=dev)
    if world > 1:
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms_total, e2e_ms_total = float(mx[0]), float(mx[1])
        E_all, graphs_all = float(sm[2]), float(sm[3])
    else:
        E_all, graphs_all = float(E), float(graphs)

    if rank == 0:
        ms_step = ms_total / args.steps
        value = E_all * L / (ms_step * 1e-3)
        e2e_ms = e2e_ms_total / e2e_steps
        if fwd_only:   # SURVEY 8d FWD_inf per layer: E(Fin s + 4) + 4(N+1) + N s (Fin + Fout)
            step_bytes = sum(E * (hdims[l] * 4 + 4) + 4 * (N + 1) + N * 4 * (hdims[l] + hdims[l + 1]) for l in range(L)) + csr_bytes(N, E)
            # cache-perfect lower bound: every source row read once (E*Fin*s -> N*Fin*s)
            step_bytes_cp = sum(4 * E + 4 * (N + 1) + N * 4 * (2 * hdims[l] + hdims[l + 1]) for l in range(L)) + csr_bytes(N, E)
        elif bf16:
            step_bytes = sum(layer_bytes_fwd_bwd_bf16feat(N, E, hdims[l], hdims[l + 1]) for l in range(L)) + csr_bytes(N, E)
            step_bytes_cp = step_bytes - sum((E - N) * (2 * hdims[l] + 4 * hdims[l]) for l in range(L))
        else:
            step_bytes = sum(layer_bytes_fwd_bwd(N, E, hdims[l], hdims[l + 1]) for l in range(L)) + csr_bytes(N, E)
            step_bytes_cp = sum(layer_bytes_fwd_bwd_cache_perfect(N, E, hdims[l], hdims[l + 1]) for l in range(L)) + csr_bytes(N, E)
        if kern is None:
            kern, top = {}, None
        else:
            # the dominant KERNEL: the single-kernel group with the largest ms x launches, backward kernels included
            # (layer_backward is the sequence of them and is reported under "kernels" only)
            single = [k for k in KERNEL_LAUNCHES_PER_LAYER if k in kern and "ms" in kern[k]]
            single = [k for k in single if not (fwd_only and k in ("ln_bwd", "dgrad", "wgrad", "segment_sum_bwd"))]
            top = max(single, key=lambda k: kern[k]["ms"] * KERNEL_LAUNCHES_PER_LAYER[k])
        traffic_ncu = committed_ncu_traffic(args.workload, top)
        line = {
            "metric": METRIC, "value": value, "unit": "edges/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16 features (fp32 accumulate, parameters and gradients)" if bf16 else "f32",
            "data": "synthetic",
            "config": dict(workload_config(args.workload, wl, N, E, graphs), feature_dtype=args.dtype),
            "graphs_per_sec": graphs_all / (ms_step * 1e-3),
            "clocks": clocks,
            "e2e": {"value": E_all * L / (e2e_ms * 1e-3), "unit": "edges/s",
                    "h2d_bytes_per_step": batches[0]["x_h"].numel() * batches[0]["x_h"].element_size() + batches[0]["ei_h"].numel() * 8,
                    "d2h_bytes_per_step": (N * hdims[-1] * (2 if bf16 else 4) if fwd_only else 4), "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "graphs_per_sec": graphs_all / (e2e_ms * 1e-3)},
            "host_numa_bound_cpus": numa,
            "gpu_launches": int(launches),
            "host_enqueue_ms_per_step": round(host_enqueue_ms, 3),
            "roofline": None if top is None else {
                "bound": "hbm", "kernel": top, "cuda_kernel": KERNEL_NAMES[top], "achieved": kern[top]["gbs"], "peak": peak_gbs,
                "unit": "GB/s", "frac": kern[top]["frac_hbm"], "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": kern[top]["algorithmic_bytes"], "ms_per_launch": kern[top]["ms"],
                "traffic_note": "DRAM bytes cannot be measured inside a plain run; the committed ncu --set full capture is quoted beside it",
                "traffic_ncu_committed": traffic_ncu,
                "candidates": {k: {"ms": kern[k]["ms"], "frac": kern[k]["frac_hbm"]} for k in single}},
            "roofline_step": {"bound": "hbm", "algorithmic_bytes": step_bytes, "achieved": step_bytes / ms_step / 1e6,
                              "peak": peak_gbs, "unit": "GB/s", "frac": step_bytes / ms_step / 1e6 / peak_gbs,
                              # the same step against the two other byte counts (VERDICT r1 weak #5): on block-diagonal
                              # batches the L2 absorbs the E*Fin gather re-reads, so 8d's figure flatters the step
                              "frac_cache_perfect": step_bytes_cp / ms_step / 1e6 / peak_gbs,
                              "algorithmic_bytes_cache_perfect": step_bytes_cp,
                              "frac_measured_dram": None,
                              "frac_measured_dram_note": "needs ncu dram__bytes of every kernel of the step; see profiles/ for the latest capture",
                              "model": ("SURVEY 8d FWD_inf: sum_l [E(Fin*4+4) + 4(N+1) + 4N(Fin+Fout)] + 24E + 8(N+1)" if fwd_only else
                                        "bf16 features: the tensors actually moved (bench.py layer_bytes_fwd_bwd_bf16feat) + 24E + 8(N+1)" if bf16 else
                                        "SURVEY 8d: sum_l [2E(Fin*4+4) + 4N(6Fin+5Fout) + 28N] + 24E + 8(N+1) (CSR rebuilt every step)")},
            "kernels": kern,
        }
        if cabi is not None:
            line["e2e_cabi_host"] = cabi
        if graphed is not None:
            line["cuda_graph"] = graphed
        if grad_sync is not None:
            line["grad_sync_check"] = grad_sync
            line["grad_overlap_check"] = overlap_check
        if world == 1 and args.workload == "batch" and not args.no_c4 and not bf16:
            for b in batches:                      # release the batch workload's device buffers first
                b.pop("x", None); b.pop("ei", None); b.pop("w", None)
            try:
                line["c4"] = c4_record(dev, peak_gbs)
            except Exception as exc:               # must never take the headline line down
                line["c4"] = {"error": repr(exc)[:300]}
        if world == 1 and not args.no_cpu:
            c = run_cpu(wl, steps=3, warmup=1, min_seconds=10.0)
            line["cpu_baseline"] = {"value": c["edges_per_s"], "unit": "edges/s", "cores": c["cores"], "kind": "port",
                                    "sample": c["sample"] + f", {c['iters']} timed iterations (about 10 s) after 1 warm-up",
                                    "graphs_per_sec": c["graphs_per_s"], "ms_per_step": c["ms"]}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", choices=sorted(WORKLOADS) + ["c2"], default="batch")
    ap.add_argument("--c2-graphs", type=int, default=1024, help="--workload c2: sequences (vehicle graphs) per GPU and step")
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--dtype", choices=["f32", "bf16"], default="f32",
                    help="f32 (default, the parity path) or bf16 FEATURE storage (x / agg / layer outputs in bf16; parameters, "
                         "accumulation, LayerNorm statistics and the whole gradient path stay fp32) -- BASELINE configs[4]")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-c4", action="store_true", help="skip the c4 sub-record of the default line")
    ap.add_argument("--skip-kernel-timing", action="store_true",
                    help="skip the per-kernel-group timing (used for the ncu launch list: only whole steps are launched)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.workload == "c2":                  # SURVEY 8(d) C2: the full GruSage training step, its own metric (bench_c2.py)
        import bench_c2
        return bench_c2.main(args)
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        main_reference(args, wl)
    else:
        main_ours(args, wl)


if __name__ == "__main__":
    main()
