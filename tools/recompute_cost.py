"""Cost of FastEGNN.recompute (FEGNN_F_RECOMPUTE, DESIGN.md 3.8): the eager training step (forward, MSE + MMD loss,
backward, FusedAdam) of bench.py's Water-3D, water3d_b20 and large (config 5: 1 M nodes, C = 8) workloads with recompute off
and on, and torch.cuda.max_memory_allocated over one step of each, at n_layers = 4, plus water3d_b20 at n_layers = 8.  The
two settings alternate block by block in one process; each block is bench.timed (CUDA events around each call, L2
overwritten before each call).  Writes one JSON file with the card name and power limit beside the numbers.

    python tools/recompute_cost.py --out profiles/recompute_cost.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from fastegnn_b200 import FastEGNN, FusedAdam, mse_mmd_loss  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def make_step(data, hp, dev, n_layers, recompute):
    torch.manual_seed(0)
    m = FastEGNN(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=64, virtual_channels=data["C"], device=dev,
                 n_layers=n_layers, gravity=data["gravity"])
    m.recompute = recompute
    opt = FusedAdam(m.parameters(), lr=5e-4, weight_decay=1e-12)
    t = {k: data[k].to(dev) for k in ("node_feat", "loc_0", "vel_0", "loc_t", "edge_index", "batch", "loc_mean", "edge_attr")}
    idx = bench.sample_indices(data["sizes"], hp["sample"], torch.Generator().manual_seed(0)).to(torch.int32).to(dev)

    def train_step():
        opt.zero_grad(set_to_none=True)
        x, Z = m(node_feat=t["node_feat"], node_loc=t["loc_0"], node_vel=t["vel_0"], edge_index=t["edge_index"],
                 data_batch=t["batch"], loc_mean=t["loc_mean"], edge_attr=t["edge_attr"])
        mse_mmd_loss(x, t["loc_t"], Z, idx, hp["sigma"], hp["weight"])[0].backward()
        opt.step()
    return train_step


def peak_bytes(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated(), torch.cuda.max_memory_allocated() - base


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=6, help="alternations of the two settings")
    ap.add_argument("--calls", type=int, default=20, help="timed calls per case and round (bench.timed)")
    ap.add_argument("--cases", default="water3d:4,water3d_b20:4,large:4,water3d_b20:8")
    ap.add_argument("--out", default="profiles/recompute_cost.json")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # 256 MB > the 126 MB L2
    res = {"card": card(), "what": "train_step ms per call (mean of a block of calls; median / p10 / p90 over the blocks), "
                                  "L2 overwritten before each call, recompute off and on alternated block by block in one "
                                  "process; train_step = forward + mse_mmd_loss + backward + FusedAdam (eager, per-call "
                                  "CsrGraph).  peak_GB = torch.cuda.max_memory_allocated over one step (model, optimizer "
                                  "and inputs included); step_GB = that less what was allocated before the step"}
    for case in args.cases.split(","):
        name, L = case.split(":")
        L = int(L)
        data, hp = bench.make_workload(name, 0, 0)
        steps = {mode: make_step(data, hp, dev, L, mode == "recompute") for mode in ("default", "recompute")}
        calls_n = max(2, args.calls // 10) if name == "large" else args.calls
        times = {mode: [] for mode in steps}
        row = {}
        for mode, fn in steps.items():
            fn()
            peak, step = peak_bytes(fn)
            row[f"peak_GB_{mode}"] = peak / 1e9
            row[f"step_GB_{mode}"] = step / 1e9
        for r in range(args.rounds + 1):            # round 0 warms every case up
            for mode, fn in steps.items():
                tm = bench.timed(fn, calls_n, flush)
                if r > 0:
                    times[mode].append(tm)
        for mode, tm in times.items():
            tm = np.array(tm)
            row[f"step_ms_{mode}"] = {"median_ms": float(np.median(tm)), "p10_ms": float(np.percentile(tm, 10)),
                                      "p90_ms": float(np.percentile(tm, 90))}
        row["time_ratio"] = row["step_ms_recompute"]["median_ms"] / row["step_ms_default"]["median_ms"]
        res[f"{name}_L{L}"] = dict(nodes=int(data["loc_0"].size(0)), graphs=int(data["n_graphs"]),
                                   edges=int(data["edge_index"].size(1)), C=int(data["C"]), n_layers=L, **row)
        print(name, L, json.dumps(row), flush=True)
        del steps
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
