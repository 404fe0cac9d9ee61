#!/usr/bin/env python
"""Long sequences and wide inputs (the projected path of csrc/gru.cu: k_gru_xproj feeds layer 0 through gi) against
torch's library GRU as GruSage._last_hidden runs it (ATen's native per-step GEMM + cell path, cuDNN disabled).

    python tools/bench_gru_long.py --out profiles/r04_gru_long.json

Three parts, all timed with CUDA events after warm-up, the paths' calls alternating (same structure as
tools/bench_gru_stack.py):
  head    -- gru(x)[1][-1] alone at N = 205 587 sequences (the C2 shape), hidden 96, L = 1 and 2, inference forward and
             forward + backward, with the max |difference| of h and the max relative difference of the parameter
             gradients against the library on the timed inputs, and the peak allocated memory of one training pass:
               T=64, I=6  and T=16, I=16 -- beyond the x tile: projected path vs library;
               T=16, I=6  -- inside the tile: tile path vs projected path (called directly) vs library, what
                             materialising gi costs where both fused paths apply.
             Every training buffer (gi / dgh / dgi 15 GB each at T = 64) is far beyond the 126 MB L2.
  kernels -- torch.profiler (a run of its own) over one projected L = 1 forward + backward at T=64, I=6: per-kernel
             device time; for k_gru_xproj and k_gru_xwgrad the achieved bytes/s from the algorithmic bytes, against the
             7.7 TB/s HBM3e figure of NVIDIA's B200 data sheet (a data-sheet figure, not a measured peak).
  c2_step -- bench_c2's model, map and batch builders with 64 frames per sequence: the eager training step at 1024
             sequence graphs, fused vs SLDM_DISABLE_FUSED_GRU=1.
The card's name, power limit and max SM clock are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import sys
import time

os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")   # 15-25 GB buffers of varying shapes
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from bench_gru_stack import gpu_info, summary, timed_alternating  # noqa: E402

N_C2, H = 205587, 96
HEAD_SHAPES = ((64, 6), (16, 16), (16, 6))
HBM_DATASHEET_TB_S = 7.7


def library_head(gru, x):
    """torch's GRU as GruSage._last_hidden runs it: cuDNN off, in slices of at most 2^30 gate elements."""
    n, rows = x.size(0), max(1, (1 << 30) // (x.size(1) * 3 * gru.hidden_size))
    with torch.backends.cudnn.flags(enabled=False):
        if n <= rows:
            return gru(x)[1][-1]
        return torch.cat([gru(x[i:i + rows])[1][-1] for i in range(0, n, rows)], dim=0)


def projected_head(gru, x):
    from sldm_gnn_b200.gru import gru_projected_last_hidden
    return gru_projected_last_hidden(gru, x)


def tile_head(gru, x):
    from sldm_gnn_b200.gru import gru_last_hidden, gru_stack_last_hidden
    return gru_last_hidden(gru, x) if gru.num_layers == 1 else gru_stack_last_hidden(gru, x)


def bench_head(dev, reps):
    from sldm_gnn_b200.gru import fused_gru_projected_eligible, fused_gru_stack_eligible
    out = {}
    for T, I in HEAD_SHAPES:
        torch.manual_seed(T * 100 + I)
        x = torch.randn(N_C2, T, I, device=dev)
        up = torch.randn(N_C2, H, device=dev)
        for L in (1, 2):
            torch.manual_seed(L)
            gru = torch.nn.GRU(I, H, L, batch_first=True).to(dev)
            assert fused_gru_projected_eligible(gru, x)
            paths = {"projected": projected_head, "library": library_head}
            if fused_gru_stack_eligible(gru, x):
                paths = {"tile": tile_head, **paths}
            res = {"tile_eligible": "tile" in paths}

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

            t = timed_alternating({k: infer(fn) for k, fn in paths.items()}, reps)
            res["forward_inference"] = {k: summary(v) for k, v in t.items()}
            t = timed_alternating({k: train(fn) for k, fn in paths.items()}, reps)
            res["forward_backward"] = {k: summary(v) for k, v in t.items()}
            for k in ("forward_inference", "forward_backward"):
                lib_ms = res[k]["library"]["median_ms"]
                res[k]["speedup_vs_library"] = {p: round(lib_ms / res[k][p]["median_ms"], 3) for p in paths if p != "library"}
            # outputs on the timed inputs and the peak memory of one training pass, per path
            outs, res["peak_allocated_gb"] = {}, {}
            for p, fn in paths.items():
                gru.zero_grad(set_to_none=True)
                torch.cuda.synchronize()
                torch.cuda.empty_cache()
                torch.cuda.reset_peak_memory_stats()
                h = fn(gru, x)
                h.backward(up)
                torch.cuda.synchronize()
                res["peak_allocated_gb"][p] = round(torch.cuda.max_memory_allocated() / 1e9, 2)
                outs[p] = (h.detach(), {k: q.grad.clone() for k, q in gru.named_parameters()})
                del h
            h_l, g_l = outs["library"]
            res["vs_library"] = {}
            for p in paths:
                if p == "library":
                    continue
                h_p, g_p = outs[p]
                res["vs_library"][p] = {
                    "max_abs_diff_h": float((h_p - h_l).abs().max()),
                    "max_rel_diff_grad": max(float((g_p[k] - g_l[k]).abs().max() / g_l[k].abs().max()) for k in g_l)}
            out[f"T{T}_I{I}_L{L}"] = res
            del gru, outs, h_l, g_l
            torch.cuda.empty_cache()
            print(f"head T={T} I={I} L={L}: {json.dumps(res)}", flush=True)
        del x, up
        torch.cuda.empty_cache()
    return out


def bench_kernels(dev):
    from torch.profiler import ProfilerActivity, profile
    T, I = 64, 6
    torch.manual_seed(0)
    x = torch.randn(N_C2, T, I, device=dev)
    up = torch.randn(N_C2, H, device=dev)
    gru = torch.nn.GRU(I, H, 1, batch_first=True).to(dev)
    for _ in range(2):
        gru.zero_grad(set_to_none=True)
        projected_head(gru, x).backward(up)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        gru.zero_grad(set_to_none=True)
        projected_head(gru, x).backward(up)
        torch.cuda.synchronize()
    rows = N_C2 * T
    nbytes = {"k_gru_xproj<96>": 4.0 * rows * (I + 3 * H),        # read x, write gi
              "k_gru_xwgrad<96>": 4.0 * rows * (3 * H + I)}       # read dgi and x (one 8-wide panel at I = 6)
    what = {"k_gru_xproj<96>": "layer-0 input projection gi = x W_ih^T + b_ih",
            "k_gru_xwgrad<96>": "layer-0 dW_ih = dgi^T x",
            "k_gru_fwd<96, true, true>": "recurrence (gi input), training",
            "k_gru_bwd<96, true>": "reverse recurrence (deep mode)",
            "k_gru_wgrad<96>": "dW_hh"}
    out = {}
    for e in prof.key_averages():
        m = re.search(r"(k_gru_\w+<[^>]*>)", e.key)
        if not m:
            continue
        name = m.group(1)
        t_us = e.device_time_total / max(e.count, 1)
        rec = {"launches": e.count, "ms_per_launch": round(t_us / 1e3, 4), "what": what.get(name)}
        if name in nbytes:
            rate = nbytes[name] / (t_us * 1e-6) / 1e12
            rec["algorithmic_gb"] = round(nbytes[name] / 1e9, 3)
            rec["achieved_tb_s"] = round(rate, 3)
            rec["of_datasheet_hbm"] = round(rate / HBM_DATASHEET_TB_S, 3)
        out[name] = rec
    print(f"kernels: {json.dumps(out)}", flush=True)
    return out


def bench_c2_step(dev, reps):
    import bench_c2 as bc
    import sldm_gnn_b200 as sg
    T = 64
    bc.T_FRAMES = T          # make_batch reads the module's frame count
    kw = dict(bc.MODEL_KW, frames_num=T)
    out = {"model": f"bench_c2.MODEL_KW with frames_num={T}"}

    def set_fused(on):
        if on:
            os.environ.pop("SLDM_DISABLE_FUSED_GRU", None)
        else:
            os.environ["SLDM_DISABLE_FUSED_GRU"] = "1"

    G = 1024
    torch.manual_seed(0)
    model = sg.GruSage(**kw, map_tensors=bc.make_map()).to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=bc.LR, weight_decay=bc.WD)
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(bc.POS_WEIGHT, device=dev))
    batches = []
    for j in range(2):
        d, N, E = bc.make_batch(G, j)
        batches.append(bc.Bag({k: v.to(dev) for k, v in d.items()}, G))
    out["eager_1024"] = {"graphs": G, "sequences": int(batches[0].x.size(0)), "frames": T}

    def eager(on, steps=3):
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
    out["eager_1024"].update({k: {kk: (round(vv / 3, 3) if kk.endswith("_ms") else vv) for kk, vv in summary(v).items()}
                              for k, v in t.items()})
    out["eager_1024"]["unit"] = "ms per step (3 steps per timed call)"
    out["eager_1024"]["speedup"] = round(out["eager_1024"]["library"]["median_ms"] / out["eager_1024"]["fused"]["median_ms"], 3)
    for name, on in (("fused", True), ("library", False)):
        set_fused(on)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats()
        eager(on, steps=1)()
        torch.cuda.synchronize()
        out["eager_1024"].setdefault("peak_allocated_gb", {})[name] = round(torch.cuda.max_memory_allocated() / 1e9, 2)
    set_fused(True)
    print(f"c2: {json.dumps(out)}", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_gru_long.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parts", default="head,kernels,c2")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "tools/bench_gru_long.py measures the B200 kernels: it needs a GPU"
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(), "torch": torch.__version__, "date": time.strftime("%Y-%m-%d"),
           "head": {"N": N_C2, "H": H, "shapes_T_I": HEAD_SHAPES},
           "library_path": "torch.nn.GRU with cuDNN disabled (ATen native per-step GEMM + cell), as GruSage._last_hidden",
           "timing": "CUDA events after warm-up, the paths' calls alternating; median over --reps"}
    parts = args.parts.split(",")
    if "head" in parts:
        res["head"]["results"] = bench_head(dev, args.reps)
    if "kernels" in parts:
        res["kernels_T64_I6_L1_forward_backward"] = bench_kernels(dev)
    if "c2" in parts:
        res["c2_step_64_frames"] = bench_c2_step(dev, args.reps)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
