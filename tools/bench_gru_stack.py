#!/usr/bin/env python
"""Stacked GRU head (GruSage(gru_num_layers = L)): the fused kernels of csrc/gru.cu against torch's library GRU as
GruSage._last_hidden runs it (ATen's native per-step GEMM + cell path, cuDNN disabled).

    python tools/bench_gru_stack.py --out profiles/r03_gru_stack.json

Three parts, all timed with CUDA events after warm-up, fused and library runs alternating:
  head    -- gru(x)[1][-1] alone at the C2 shape (205 587 sequences x 16 frames x 6 features, hidden 96), L = 1, 2, 3:
             inference forward and forward + backward, with the max |difference| of h and of every parameter
             gradient between the two paths on the timed inputs.  x is 79 MB, but the per-layer buffers of a
             training pass (saved gates 6.3 GB, gi / dgh / dgi 3.8 GB each) are far beyond the 126 MB L2.
  kernels -- torch.profiler (a run of its own) over one fused L = 2 forward + backward: per-kernel device time and the
             achieved FP32 rate from the algorithmic flops, against the FFMA ceilings of profiles/r01m_ffma2_probe.txt.
  c2_step -- bench_c2's model, map and batches with gru_num_layers = 2: the eager training step at 1024 sequence graphs
             and GraphedTrainStep at 32, fused vs SLDM_DISABLE_FUSED_GRU=1.
The card's name, power limit and max SM clock are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

N_C2, T_C2, I_C2, H_C2 = 205587, 16, 6, 96
# profiles/r01m_ffma2_probe.txt (B200, 148 SMs): independent FFMA chains, and the register-tiled 8 x 9 outer product
FFMA_CEILINGS = {"ffma_chains": 66.3, "ffma_outer_product_8x9": 56.3, "ffma2_outer_product_8x9": 65.4}


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in out.stdout.splitlines()[0].split(",")])) if out.stdout else {}


def library_head(gru, x):
    with torch.backends.cudnn.flags(enabled=False):
        return gru(x)[1][-1]


def fused_head(gru, x):
    from sldm_gnn_b200.gru import gru_last_hidden, gru_stack_last_hidden
    return gru_last_hidden(gru, x) if gru.num_layers == 1 else gru_stack_last_hidden(gru, x)


def timed_alternating(fns, reps, warmup=2):
    """fns: {name: callable}; each is warmed up, then the calls alternate; returns {name: [ms per call]}."""
    for fn in fns.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    res = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            res[k].append(a.elapsed_time(b))
    return res


def summary(ms):
    s = sorted(ms)
    return {"median_ms": round(s[len(s) // 2], 3), "min_ms": round(s[0], 3), "max_ms": round(s[-1], 3), "n": len(s)}


def bench_head(dev, reps):
    out = {}
    torch.manual_seed(0)
    x = torch.randn(N_C2, T_C2, I_C2, device=dev)
    up = torch.randn(N_C2, H_C2, device=dev)
    for L in (1, 2, 3):
        torch.manual_seed(L)
        gru = torch.nn.GRU(I_C2, H_C2, L, batch_first=True).to(dev)
        res = {}

        def infer(fn):
            def run():
                with torch.no_grad():
                    return fn(gru, x)
            return run

        def train(fn):
            def run():
                gru.zero_grad(set_to_none=True)
                fn(gru, x).backward(up)
            return run

        t = timed_alternating({"fused": infer(fused_head), "library": infer(library_head)}, reps)
        res["forward_inference"] = {k: summary(v) for k, v in t.items()}
        t = timed_alternating({"fused": train(fused_head), "library": train(library_head)}, reps)
        res["forward_backward"] = {k: summary(v) for k, v in t.items()}
        for k in ("forward_inference", "forward_backward"):
            res[k]["speedup"] = round(res[k]["library"]["median_ms"] / res[k]["fused"]["median_ms"], 3)
        # outputs of the two paths on the timed inputs
        gru.zero_grad(set_to_none=True)
        h_f = fused_head(gru, x)
        h_f.backward(up)
        g_f = {k: p.grad.clone() for k, p in gru.named_parameters()}
        gru.zero_grad(set_to_none=True)
        h_l = library_head(gru, x)
        h_l.backward(up)
        res["max_abs_diff"] = {"h": float((h_f - h_l).abs().max())}
        res["max_abs_diff"].update({f"grad_{k}": float((g_f[k] - p.grad).abs().max()) for k, p in gru.named_parameters()})
        res["max_abs_grad"] = {f"grad_{k}": float(p.grad.abs().max()) for k, p in gru.named_parameters()}
        out[f"L{L}"] = res
        del gru, h_f, h_l, g_f
        torch.cuda.empty_cache()
        print(f"head L={L}: {json.dumps(res)}", flush=True)
    return out


def bench_kernels(dev):
    from torch.profiler import ProfilerActivity, profile
    torch.manual_seed(0)
    x = torch.randn(N_C2, T_C2, I_C2, device=dev)
    up = torch.randn(N_C2, H_C2, device=dev)
    gru = torch.nn.GRU(I_C2, H_C2, 2, batch_first=True).to(dev)
    for _ in range(2):
        gru.zero_grad(set_to_none=True)
        fused_head(gru, x).backward(up)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        gru.zero_grad(set_to_none=True)
        fused_head(gru, x).backward(up)
        torch.cuda.synchronize()
    rows, H = N_C2 * T_C2, H_C2
    gemm = 2.0 * rows * 3 * H * H            # one [rows] x [H] x [3H] product
    flops = {"k_gru_fwd<96, true, false>": gemm + 2.0 * rows * 3 * H * I_C2, "k_gru_fwd<96, true, true>": gemm,
             "k_gru_proj<96, true>": gemm, "k_gru_proj<96, false>": gemm, "k_gru_bwd<96, false>": gemm,
             "k_gru_bwd<96, true>": gemm, "k_gru_wgrad<96>": gemm}
    what = {"k_gru_fwd<96, true, false>": "layer 0 recurrence (x tile), training",
            "k_gru_fwd<96, true, true>": "layer 1 recurrence (gi input), training",
            "k_gru_proj<96, true>": "input projection gi = h_seq W_ih^T + b_ih",
            "k_gru_proj<96, false>": "data gradient dY = dgi W_ih",
            "k_gru_bwd<96, false>": "layer 0 reverse recurrence", "k_gru_bwd<96, true>": "layer 1 reverse recurrence",
            "k_gru_wgrad<96>": "dW_hh (both layers) and dW_ih of layer 1, per launch"}
    out = {}
    for e in prof.key_averages():
        m = re.search(r"(k_gru_\w+<[^>]*>)", e.key)
        if not m:
            continue
        name = m.group(1)
        t_us = e.device_time_total / max(e.count, 1)
        rec = {"launches": e.count, "ms_per_launch": round(t_us / 1e3, 4), "what": what.get(name)}
        if name in flops:
            tf = flops[name] / (t_us * 1e-6) / 1e12
            rec["algorithmic_tflops"] = round(flops[name] / 1e12, 4)
            rec["achieved_tflop_s"] = round(tf, 2)
            rec["of_ffma_ceilings"] = {k: round(tf / v, 3) for k, v in FFMA_CEILINGS.items()}
        out[name] = rec
    print(f"kernels: {json.dumps(out)}", flush=True)
    return out


def bench_c2_step(dev, reps):
    import torch.nn.functional as Fn
    import bench_c2 as bc
    import sldm_gnn_b200 as sg
    from sldm_gnn_b200.grusage import GraphedTrainStep
    kw = dict(bc.MODEL_KW, gru_num_layers=2)
    out = {"model": "bench_c2.MODEL_KW with gru_num_layers=2"}

    def set_fused(on):
        if on:
            os.environ.pop("SLDM_DISABLE_FUSED_GRU", None)
        else:
            os.environ["SLDM_DISABLE_FUSED_GRU"] = "1"

    # eager step at 1024 sequence graphs
    G = 1024
    torch.manual_seed(0)
    model = sg.GruSage(**kw, map_tensors=bc.make_map()).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=bc.LR, weight_decay=bc.WD)
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(bc.POS_WEIGHT, device=dev))
    batches = []
    for j in range(2):
        d, N, E = bc.make_batch(G, j)
        batches.append(bc.Bag({k: v.to(dev) for k, v in d.items()}, G))
    out["eager_1024"] = {"graphs": G, "sequences": int(batches[0].x.size(0))}

    def eager(on, steps=5):
        def run():
            set_fused(on)
            for i in range(steps):
                opt.zero_grad()
                loss = crit(model(batches[i % 2]), batches[i % 2].y)
                loss.backward()
                opt.step()
                loss.item()
        return run

    t = timed_alternating({"fused": eager(True), "library": eager(False)}, reps)
    out["eager_1024"].update({k: {kk: (round(vv / 5, 3) if kk.endswith("_ms") else vv) for kk, vv in summary(v).items()}
                              for k, v in t.items()})
    out["eager_1024"]["unit"] = "ms per step (5 steps per timed call)"
    out["eager_1024"]["speedup"] = round(out["eager_1024"]["library"]["median_ms"] / out["eager_1024"]["fused"]["median_ms"], 3)
    set_fused(True)
    del model, opt, batches
    torch.cuda.empty_cache()

    # GraphedTrainStep at 32 sequence graphs: the path is fixed when the step is captured
    G = 32
    torch.manual_seed(0)
    base = sg.GruSage(**kw, map_tensors=bc.make_map()).to(dev)
    batches = []
    for j in range(2):
        d, N, E = bc.make_batch(G, j)
        batches.append(bc.Bag({k: v.to(dev) for k, v in d.items()}, G))
    pw = torch.tensor(bc.POS_WEIGHT, device=dev)
    steps = {}
    for name, on in (("fused", True), ("library", False)):
        set_fused(on)
        m = copy.deepcopy(base)
        o = torch.optim.Adam(m.parameters(), lr=bc.LR, weight_decay=bc.WD, capturable=True, fused=True)
        ts = GraphedTrainStep(m, o, lambda lg, y, w: Fn.binary_cross_entropy_with_logits(lg, y, weight=w, pos_weight=pw, reduction="sum"),
                              max_nodes=max(b.x.size(0) for b in batches) + 1,
                              max_edges=max(b.edge_index.size(1) for b in batches), max_graphs=G + 1)
        for i in range(3):
            ts(batches[i % 2], batches[i % 2].y).item()
        steps[name] = ts
    set_fused(True)

    def graphed(ts, n=50):
        def run():
            for i in range(n):
                ts(batches[i % 2], batches[i % 2].y).item()
        return run

    t = timed_alternating({k: graphed(v) for k, v in steps.items()}, reps)
    out["graphed_train_step_32"] = {k: {kk: (round(vv / 50, 4) if kk.endswith("_ms") else vv) for kk, vv in summary(v).items()}
                                    for k, v in t.items()}
    out["graphed_train_step_32"]["unit"] = "ms per step (50 steps per timed call)"
    out["graphed_train_step_32"]["speedup"] = round(out["graphed_train_step_32"]["library"]["median_ms"]
                                                    / out["graphed_train_step_32"]["fused"]["median_ms"], 3)
    print(f"c2: {json.dumps(out)}", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_gru_stack.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parts", default="head,kernels,c2")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tools/bench_gru_stack.py measures the B200 kernels: it needs a GPU"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(), "torch": torch.__version__, "date": time.strftime("%Y-%m-%d"),
           "head_shape": {"N": N_C2, "T": T_C2, "I": I_C2, "H": H_C2},
           "library_path": "torch.nn.GRU with cuDNN disabled (ATen native per-step GEMM + cell), as GruSage._last_hidden",
           "timing": "CUDA events after warm-up, fused and library calls alternating; median over --reps"}
    parts = args.parts.split(",")
    if "head" in parts:
        res["head"] = bench_head(dev, args.reps)
    if "kernels" in parts:
        res["kernels_L2_forward_backward"] = bench_kernels(dev)
        res["ffma_ceilings_tflop_s"] = dict(FFMA_CEILINGS, source="profiles/r01m_ffma2_probe.txt")
    if "c2" in parts:
        res["c2_step_two_layers"] = bench_c2_step(dev, args.reps)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
