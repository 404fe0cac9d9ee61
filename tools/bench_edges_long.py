#!/usr/bin/env python
"""Proximity-edge construction (csrc/edge_build.cu) at windows of 16 to 4096 frames, against the reference's loop.

    python tools/bench_edges_long.py --out profiles/r06_edges_long.json [--parent-src FILE.cu]

  shapes    -- V = 300 and 1000 vehicles, T = 16, 128, 256, 1024, 4096 frames: one `build_proximity_edges` call (count
               pass, the host read of the edge count, fill pass) timed with CUDA events, median of --reps calls after
               warm-up, and V (V - 1) T pair-frames per second (each pass walks every ordered pair's frames once; the
               fill pass walks an edge's frames a second time for its sums).  x at V = 1000, T = 4096 is 98 MB: it
               stays in L2, which is where a window built right after its features were written finds it.
  reference -- the reference's Python double loop (oracle/edges_oracle.py) on the host, once per T at V = 300.
  parent    -- with --parent-src (an untracked copy of an earlier edge_build.cu, kept outside sldm_gnn_b200/csrc/ so the
               Makefile does not compile it too): that unit is compiled and linked with the tree's other objects into
               build/ab/edges_parent.so, the way tools/build_variant.sh builds variants, and run in a second worker
               process (SLDM_LIB_PATH).  At T = 16 and 128 the two libraries' calls alternate, --rounds rounds of
               --reps calls each, and their outputs are compared bit for bit.
Each library runs in its own worker process; this process only drives them and runs the reference loop.  The card's
name, power limit and max SM clock are read in the same run and stored with the numbers.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

VS, TS, T_AB = (300, 1000), (16, 128, 256, 1024, 4096), (16, 128)
RADIUS = 30.0


def make_x(V, T, seed=0):
    """Vehicles spread over 400 m moving at up to 2 m per frame, present 90 % of the frames."""
    import torch
    g = torch.Generator().manual_seed(seed)
    x = torch.zeros(V, T, 6)
    start = (torch.rand(V, 1, 2, generator=g) - 0.5) * 400.0
    vel = (torch.rand(V, 1, 2, generator=g) - 0.5) * 4.0
    x[:, :, :2] = start + vel * torch.arange(T).view(1, T, 1)
    x[:, :, 2] = torch.rand(V, T, generator=g) * 30
    x[:, :, 3] = torch.rand(V, T, generator=g) * 6.28
    x[:, :, 4] = (torch.rand(V, T, generator=g) < 0.9).float()
    x[:, :, 5] = torch.rand(V, T, generator=g)
    return x


def worker():
    """One JSON request per stdin line {"V", "T", "reps", "warmup"}; answers with the per-call times and a digest."""
    import torch
    import sldm_gnn_b200 as sg
    cache = {}
    for line in sys.stdin:
        req = json.loads(line)
        key = (req["V"], req["T"])
        if key not in cache:
            cache.clear()
            cache[key] = make_x(*key).cuda()
        x = cache[key]
        for _ in range(req["warmup"]):
            ei, ea = sg.build_proximity_edges(x, RADIUS)
        torch.cuda.synchronize()
        ms = []
        for _ in range(req["reps"]):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ei, ea = sg.build_proximity_edges(x, RADIUS)
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        h = hashlib.sha256(ei.cpu().numpy().tobytes() + ea.cpu().numpy().tobytes()).hexdigest()[:16]
        print(json.dumps({"ms": ms, "E": int(ei.size(1)), "digest": h}), flush=True)


class Worker:
    def __init__(self, lib=None):
        env = dict(os.environ)
        if lib:
            env["SLDM_LIB_PATH"] = lib
        self.p = subprocess.Popen([sys.executable, os.path.abspath(__file__), "--worker"], cwd=ROOT, env=env,
                                  stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)

    def run(self, V, T, reps, warmup=3):
        self.p.stdin.write(json.dumps({"V": V, "T": T, "reps": reps, "warmup": warmup}) + "\n")
        self.p.stdin.flush()
        line = self.p.stdout.readline()
        if not line:
            raise RuntimeError(f"worker exited with {self.p.wait()}")
        return json.loads(line)

    def close(self):
        self.p.stdin.close()
        self.p.wait()


def build_parent(src):
    """src compiled in place of edge_build.cu and linked with the tree's other objects -> build/ab/edges_parent.so"""
    so = os.path.join(ROOT, "build", "ab", "edges_parent.so")
    if os.path.exists(so) and os.path.getmtime(so) > os.path.getmtime(src):
        return so
    subprocess.run(["make", "-j8", "sldm_gnn_b200/lib/libsldm_sage.so"], cwd=ROOT, check=True, stdout=subprocess.DEVNULL)
    out_dir = os.path.join(ROOT, "build", "ab", "obj_edges_parent")
    os.makedirs(out_dir, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    arch = ["-gencode", "arch=compute_100a,code=sm_100a"]
    obj = os.path.join(out_dir, "edge_build.o")
    subprocess.run([nvcc, "-O3", "-std=c++17", "-lineinfo", *arch, "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
                    "-I", os.path.join(ROOT, "sldm_gnn_b200", "csrc"), "-c", src, "-o", obj], check=True)
    objs = sorted(os.path.join(ROOT, "build", "obj", f) for f in os.listdir(os.path.join(ROOT, "build", "obj"))
                  if f.endswith(".o") and f != "edge_build.o")
    subprocess.run([nvcc, "-shared", *arch, "-o", so, *objs, obj, "-cudart", "static"], check=True)
    return so


def summary(ms):
    s = sorted(ms)
    return {"median_ms": round(s[len(s) // 2], 4), "min_ms": round(s[0], 4), "max_ms": round(s[-1], 4), "n": len(s)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_edges_long.json"))
    ap.add_argument("--reps", type=int, default=21)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--parent-src", default=None)
    ap.add_argument("--worker", action="store_true")
    args = ap.parse_args()
    if args.worker:
        return worker()

    from bench_gru_stack import gpu_info
    from oracle.edges_oracle import proximity_edges_oracle
    parent_lib = build_parent(os.path.abspath(args.parent_src)) if args.parent_src else None
    res = {"gpu": gpu_info(), "radius": RADIUS, "shapes": [], "reference": [], "parent_ab": []}
    new = Worker()
    try:
        for V in VS:
            for T in TS:
                r = new.run(V, T, args.reps)
                s = summary(r["ms"])
                pf = V * (V - 1) * T
                res["shapes"].append({"V": V, "T": T, "E": r["E"], **s, "pair_frames": pf,
                                      "pair_frames_per_s": round(pf / (s["median_ms"] * 1e-3), 1)})
                print(json.dumps(res["shapes"][-1]), flush=True)
        for T in TS:
            V = 300
            x = make_x(V, T)
            t0 = time.perf_counter()
            ei, _ = proximity_edges_oracle(x, RADIUS)
            ref_ms = (time.perf_counter() - t0) * 1e3
            dev_ms = next(s["median_ms"] for s in res["shapes"] if s["V"] == V and s["T"] == T)
            res["reference"].append({"V": V, "T": T, "E": int(ei.size(1)), "reference_loop_ms": round(ref_ms, 1),
                                     "device_ms": dev_ms, "speedup": round(ref_ms / dev_ms, 1)})
            print(json.dumps(res["reference"][-1]), flush=True)
        if parent_lib:
            old = Worker(parent_lib)
            try:
                for V in VS:
                    for T in T_AB:
                        ms = {"new": [], "parent": []}
                        dig = {}
                        for _ in range(args.rounds):
                            for name, w in (("new", new), ("parent", old)):
                                r = w.run(V, T, args.reps // 3 or 1, warmup=2)
                                ms[name] += r["ms"]
                                dig[name] = r["digest"]
                        row = {"V": V, "T": T, "new": summary(ms["new"]), "parent": summary(ms["parent"]),
                               "outputs_equal": dig["new"] == dig["parent"]}
                        row["new_over_parent"] = round(row["new"]["median_ms"] / row["parent"]["median_ms"], 3)
                        res["parent_ab"].append(row)
                        print(json.dumps(row), flush=True)
            finally:
                old.close()
    finally:
        new.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
