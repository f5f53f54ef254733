"""Cost of fegnn_set_mode("layer_overlap"): the eager FastEGNN training step (forward, MSE + MMD loss, backward, FusedAdam)
and the backward alone of bench.py's Water-3D, water3d_b20 and large (1 M nodes) workloads with the mode at 2 (on at
every size) and 0 (off).  The two settings alternate block by block in one process; each block is bench.timed (CUDA events around each call, L2
overwritten before each call).  Writes one JSON file with the card name and power limit beside the numbers.

    python tools/layer_overlap_cost.py --out profiles/layer_overlap_cost.json
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
from fastegnn_b200 import FastEGNN, FusedAdam, _lib, mse_mmd_loss  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def make_calls(data, hp, dev):
    torch.manual_seed(0)
    m = FastEGNN(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=64, virtual_channels=data["C"], device=dev, n_layers=4,
                 gravity=data["gravity"])
    opt = FusedAdam(m.parameters(), lr=5e-4, weight_decay=1e-12)
    t = {k: data[k].to(dev) for k in ("node_feat", "loc_0", "vel_0", "loc_t", "edge_index", "batch", "loc_mean", "edge_attr")}
    idx = bench.sample_indices(data["sizes"], hp["sample"], torch.Generator().manual_seed(0)).to(torch.int32).to(dev)

    def forward():
        x, Z = m(node_feat=t["node_feat"], node_loc=t["loc_0"], node_vel=t["vel_0"], edge_index=t["edge_index"],
                 data_batch=t["batch"], loc_mean=t["loc_mean"], edge_attr=t["edge_attr"])
        return mse_mmd_loss(x, t["loc_t"], Z, idx, hp["sigma"], hp["weight"])[0]

    def train_step():
        opt.zero_grad(set_to_none=True)
        forward().backward()
        opt.step()
    loss = forward()

    def backward():
        loss.backward(retain_graph=True)
    return {"train_step": train_step, "backward": backward}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=6, help="alternations of the two settings")
    ap.add_argument("--calls", type=int, default=20, help="timed calls per case and round (bench.timed)")
    ap.add_argument("--workloads", default="water3d,water3d_b20,large")
    ap.add_argument("--out", default="profiles/layer_overlap_cost.json")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # 256 MB > the 126 MB L2
    res = {"card": card(), "what": "ms per call (mean of a block of calls; median / p10 / p90 over the blocks), L2 "
                                  "overwritten before each call, layer_overlap 2 and 0 alternated block by block in one "
                                  "process; train_step = forward + mse_mmd_loss + backward + FusedAdam (eager, per-call "
                                  "CsrGraph); backward = loss.backward of a kept graph"}
    old = _lib.get_mode("layer_overlap")
    for name in args.workloads.split(","):
        data, hp = bench.make_workload(name, 0, 0)
        calls = make_calls(data, hp, dev)
        calls_n = max(2, args.calls // 10) if name == "large" else args.calls
        times = {f"{k}_{mode}": [] for k in calls for mode in ("on", "off")}
        for r in range(args.rounds + 1):            # round 0 warms every case up
            for mode in ("on", "off"):
                _lib.set_mode("layer_overlap", 2 if mode == "on" else 0)
                for k, fn in calls.items():
                    tm = bench.timed(fn, calls_n, flush)
                    if r > 0:
                        times[f"{k}_{mode}"].append(tm)
        _lib.set_mode("layer_overlap", old)
        row = {}
        for k, tm in times.items():
            tm = np.array(tm)
            row[k] = {"median_ms": float(np.median(tm)), "p10_ms": float(np.percentile(tm, 10)),
                      "p90_ms": float(np.percentile(tm, 90))}
        res[name] = dict(nodes=int(data["loc_0"].size(0)), graphs=int(data["n_graphs"]),
                         edges=int(data["edge_index"].size(1)), **row)
        print(name, json.dumps(row), flush=True)
        del calls
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
