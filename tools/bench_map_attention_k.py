#!/usr/bin/env python
"""Map attention at K = 5..32 nearest segments (csrc/map_attention.cu: per-thread lists up to K = 8, one warp per
vehicle above) against the reference's op chain (the oracle, plain torch, on the GPU).

    python tools/bench_map_attention_k.py --out profiles/r05_map_attention_k.json

Two parts, timed with CUDA events after warm-up, the calls of one configuration alternating, median of --reps:
  attention -- MapSpatialAttention alone on a 2048-segment map (bench_c2's centroids), B = 205 587 (the C2 step's vehicles
               at 1024 graphs) and 821 772, D = 8 and 32, K = 5, 8, 9, 16, 32: the grid forward (the default), the
               exhaustive-scan forward (SLDM_MAP_ATTENTION_SCAN=1) and the backward for the embeddings and the MLP,
               membership CSR build included.  Beside the times, the algorithmic bytes of each call computed from the
               shapes (`fwd_bytes`, `bwd_bytes`).  The [S, D] table (at most 256 KB) stays in L2, so the embedding-row
               gathers are L2 traffic, not HBM.  At B = 205 587 the reference's op chain (the oracle on CUDA), forward
               and forward + backward.
  c2_step   -- bench_c2's model, map and batch builders: the eager training step at 1024 graphs with
               map_attention_topk = 5, 16 and 32.
The card's name, power limit and max SM clock are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from bench_gru_stack import gpu_info, summary, timed_alternating  # noqa: E402

S, H = 2048, 16
BS, DS, KS = (205587, 821772), (8, 32), (5, 8, 9, 16, 32)
B_REF = 205587


def fwd_bytes(B, D, K):
    """positions in, K embedding rows gathered, ctx out, idx (int64) / dist / w out"""
    return B * (8 + K * D * 4 + D * 4 + K * 16)


def bwd_bytes(B, D, K):
    """ds: dctx, idx, w and K embedding rows in, ds out; MLP: dist and ds in; membership CSR: the B*K indices in, the
    sorted member ids out (one pass each way); d_emb: member ids, weights and one dctx row per member in, [S, D] out"""
    ds = B * (D * 4 + K * 12 + K * D * 4 + K * 4)
    mlp = B * K * 8
    csr = B * K * (8 + 4)
    demb = B * K * (4 + 4 + D * 4) + S * D * 4
    return ds + mlp + csr + demb


def set_scan(on):
    if on:
        os.environ["SLDM_MAP_ATTENTION_SCAN"] = "1"
    else:
        os.environ.pop("SLDM_MAP_ATTENTION_SCAN", None)


def bench_attention(dev, reps):
    import bench_c2 as bc
    import sldm_gnn_b200 as sg
    from oracle.map_attention_oracle import MapSpatialAttentionOracle
    cent = bc.make_map()["mseg_centroids"]
    rows = []
    for B in BS:
        g = torch.Generator().manual_seed(B)
        pos = (torch.rand(B, 2, generator=g) * bc.EXTENT).to(dev)
        for D in DS:
            emb = torch.randn(S, D, generator=g).to(dev)
            up = torch.randn(B, D, generator=g).to(dev)
            for K in KS:
                torch.manual_seed(K)
                m = sg.MapSpatialAttention(cent, K).to(dev)
                e = emb.clone().requires_grad_(True)
                params = [e] + list(m.parameters())
                set_scan(False)
                y = m(pos, e)

                def fwd(scan):
                    def run():
                        set_scan(scan)
                        with torch.no_grad():
                            m(pos, emb)
                    return run

                fns = {"grid_fwd": fwd(False), "scan_fwd": fwd(True),
                       "bwd": lambda: torch.autograd.grad(y, params, up, retain_graph=True)}
                ref = None
                if B == B_REF:
                    ref = MapSpatialAttentionOracle(cent.to(dev), K).to(dev)
                    ref.load_state_dict(m.state_dict(), strict=True)
                    er = emb.clone().requires_grad_(True)

                    def ref_fwd():
                        with torch.no_grad():
                            ref(pos, emb)

                    def ref_fwd_bwd():
                        torch.autograd.grad(ref(pos, er), [er] + list(ref.parameters()), up)

                    fns.update({"reference_fwd": ref_fwd, "reference_fwd_bwd": ref_fwd_bwd})
                t = timed_alternating(fns, reps)
                set_scan(False)
                row = {"B": B, "S": S, "D": D, "K": K, "fwd_bytes": fwd_bytes(B, D, K), "bwd_bytes": bwd_bytes(B, D, K)}
                row.update({k: summary(v) for k, v in t.items()})
                g_ms, b_ms = row["grid_fwd"]["median_ms"], row["bwd"]["median_ms"]
                row["grid_fwd_GB_s"] = round(row["fwd_bytes"] / (g_ms * 1e6), 1)
                row["bwd_GB_s"] = round(row["bwd_bytes"] / (b_ms * 1e6), 1)
                if ref is not None:
                    row["speedup_fwd_vs_reference"] = round(row["reference_fwd"]["median_ms"] / g_ms, 2)
                    row["speedup_fwd_bwd_vs_reference"] = round(row["reference_fwd_bwd"]["median_ms"] / (g_ms + b_ms), 2)
                print(f"attention: {json.dumps(row)}", flush=True)
                rows.append(row)
                del m, y, params, ref
                torch.cuda.empty_cache()
    return rows


def bench_c2_step(dev, reps):
    import bench_c2 as bc
    import sldm_gnn_b200 as sg
    G = 1024
    batches = []
    for j in range(2):
        d, N, E = bc.make_batch(G, j)
        batches.append(bc.Bag({k: v.to(dev) for k, v in d.items()}, G))
    models = {}
    for K in (5, 16, 32):
        torch.manual_seed(0)
        model = sg.GruSage(**dict(bc.MODEL_KW, map_attention_topk=K), map_tensors=bc.make_map()).to(dev)
        opt = torch.optim.Adam(model.parameters(), lr=bc.LR, weight_decay=bc.WD)
        models[K] = (model, opt)
    crit = torch.nn.BCEWithLogitsLoss(pos_weight=torch.tensor(bc.POS_WEIGHT, device=dev))

    def eager(K, steps=5):
        model, opt = models[K]

        def run():
            for i in range(steps):
                opt.zero_grad()
                loss = crit(model(batches[i % 2]), batches[i % 2].y)
                loss.backward()
                opt.step()
                loss.item()
        return run

    t = timed_alternating({f"top{K}": eager(K) for K in models}, reps)
    out = {"model": "bench_c2.MODEL_KW with map_attention_topk = 5, 16, 32", "graphs": G,
           "sequences": int(batches[0].x.size(0)), "unit": "ms per step (5 steps per timed call)"}
    out.update({k: {kk: (round(vv / 5, 3) if kk.endswith("_ms") else vv) for kk, vv in summary(v).items()} for k, v in t.items()})
    print(f"c2: {json.dumps(out)}", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--parts", default="attention,c2")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_map_attention_k.py measures the GPU kernels: no CUDA device found")
    dev = torch.device("cuda:0")
    parts = args.parts.split(",")
    res = {"gpu": gpu_info(), "torch": torch.__version__, "reps": args.reps,
           "timing": "CUDA events, warm-up 2 calls, calls of one configuration alternating, median"}
    if "attention" in parts:
        res["attention"] = bench_attention(dev, args.reps)
    if "c2" in parts:
        res["c2_step"] = bench_c2_step(dev, args.reps)
    text = json.dumps(res, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
