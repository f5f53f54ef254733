"""Cost of the input gradients: the eager FastEGNN training step (forward, MSE + MMD loss, backward, FusedAdam) and the
backward alone of bench.py's Water-3D and water3d_b20 workloads, with no input gradient requested and with node_vel,
edge_attr and node_attr (node_attr_nf = 4) all requested.  The cases alternate block by block in one process; each block
is bench.timed (CUDA events around each call, L2 overwritten before each call).  Writes one JSON file with the card name
and power limit beside the numbers.

    python tools/input_grads_cost.py --out profiles/input_grads_cost.json
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

FA = 4


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def make_case(data, hp, want, dev, backward_only):
    """want: request all three input gradients.  backward_only: time loss.backward() of a kept graph (retain_graph)."""
    torch.manual_seed(0)
    m = FastEGNN(node_feat_nf=2, node_attr_nf=FA, edge_attr_nf=2, hidden_nf=64, virtual_channels=data["C"], device=dev,
                 n_layers=4, gravity=data["gravity"])
    opt = FusedAdam(m.parameters(), lr=5e-4, weight_decay=1e-12)
    t = {k: data[k].to(dev) for k in ("node_feat", "loc_0", "vel_0", "loc_t", "edge_index", "batch", "loc_mean", "edge_attr")}
    a = torch.rand(t["loc_0"].size(0), FA, generator=torch.Generator().manual_seed(1)).to(dev)
    v, ea = t["vel_0"].clone().requires_grad_(want), t["edge_attr"].clone().requires_grad_(want)
    a.requires_grad_(want)
    idx = bench.sample_indices(data["sizes"], hp["sample"], torch.Generator().manual_seed(0)).to(torch.int32).to(dev)

    def forward():
        x, Z = m(node_feat=t["node_feat"], node_loc=t["loc_0"], node_vel=v, edge_index=t["edge_index"],
                 data_batch=t["batch"], loc_mean=t["loc_mean"], edge_attr=ea, node_attr=a)
        return mse_mmd_loss(x, t["loc_t"], Z, idx, hp["sigma"], hp["weight"])[0]

    if backward_only:
        loss = forward()

        def call():
            loss.backward(retain_graph=True)
        return call

    def call():
        opt.zero_grad(set_to_none=True)
        for p in (v, ea, a):
            p.grad = None
        forward().backward()
        opt.step()
    return call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=8, help="alternations of the cases")
    ap.add_argument("--calls", type=int, default=20, help="timed calls per case and round (bench.timed)")
    ap.add_argument("--out", default="profiles/input_grads_cost.json")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # 256 MB > the 126 MB L2
    res = {"card": card(), "what": "ms per call (mean of a block of calls; median / p10 / p90 over the blocks), L2 "
                                  "overwritten before each call, cases alternated block by block in one process; "
                                  f"train_step = forward + mse_mmd_loss + backward + FusedAdam (eager, node_attr_nf = {FA}, "
                                  "edge_attr_nf = 2, per-call CsrGraph); backward = loss.backward of a kept graph; "
                                  "'none' requests no input gradient, 'all' requests node_vel, edge_attr and node_attr"}
    for name in ("water3d", "water3d_b20"):
        data, hp = bench.make_workload(name, 0, 0)
        cases = {f"{what}_{req}": make_case(data, hp, req == "all", dev, what == "backward")
                 for what in ("train_step", "backward") for req in ("none", "all")}
        times = {k: [] for k in cases}
        for r in range(args.rounds + 1):            # round 0 warms every case up
            for k, fn in cases.items():
                t = bench.timed(fn, args.calls, flush)
                if r > 0:
                    times[k].append(t)
        row = {}
        for k, t in times.items():
            t = np.array(t)
            row[k] = {"median_ms": float(np.median(t)), "p10_ms": float(np.percentile(t, 10)),
                      "p90_ms": float(np.percentile(t, 90))}
        res[name] = dict(nodes=int(data["loc_0"].size(0)), graphs=int(data["n_graphs"]), edges=int(data["edge_index"].size(1)),
                         **row)
        print(name, json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
