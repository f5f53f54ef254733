"""Cost of node attributes: the FastEGNN training step (forward, MSE + MMD loss, backward, FusedAdam) of bench.py's
Water-3D and water3d_b20 workloads at node_attr_nf = 0, 1 and 16, and fegnn_node_pre_forward + _backward of one layer
alone, the cases alternated in one process: bench.timed (CUDA events around each call, L2 overwritten before each call)
over blocks of calls, the cases taking turns block by block.  Writes one JSON file with the card name and power limit
beside the numbers.

    python tools/node_attr_cost.py --out profiles/node_attr_cost.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from fastegnn_b200 import FastEGNN, FusedAdam, _lib as L, mse_mmd_loss  # noqa: E402
from fastegnn_b200.ops import CsrGraph, SavedBlock, layer_ptrs, make_dims  # noqa: E402

WIDTHS = (0, 1, 16)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def step_case(data, hp, Fa, dev):
    torch.manual_seed(0)
    m = FastEGNN(node_feat_nf=2, node_attr_nf=Fa, edge_attr_nf=2, hidden_nf=64, virtual_channels=data["C"], device=dev,
                 n_layers=4, gravity=data["gravity"])
    opt = FusedAdam(m.parameters(), lr=5e-4, weight_decay=1e-12)
    t = {k: data[k].to(dev) for k in ("node_feat", "loc_0", "vel_0", "loc_t", "edge_index", "batch", "loc_mean", "edge_attr")}
    a = torch.rand(t["loc_0"].size(0), Fa, generator=torch.Generator().manual_seed(1)).to(dev) if Fa else None
    idx = bench.sample_indices(data["sizes"], hp["sample"], torch.Generator().manual_seed(0)).to(torch.int32).to(dev)
    graph = CsrGraph(t["edge_index"], t["batch"], t["edge_attr"], data["n_graphs"])

    def call():
        opt.zero_grad(set_to_none=True)
        x, Z = m(node_feat=t["node_feat"], node_loc=t["loc_0"], node_vel=t["vel_0"], edge_index=graph,
                 data_batch=t["batch"], loc_mean=t["loc_mean"], node_attr=a)
        loss, _ = mse_mmd_loss(x, t["loc_t"], Z, idx, hp["sigma"], hp["weight"])
        loss.backward()
        opt.step()
    return call


def node_pre_case(data, Fa, dev):
    """fegnn_node_pre_forward + fegnn_node_pre_backward of a (not last) layer with gravity, default modes."""
    torch.manual_seed(0)
    m = FastEGNN(node_feat_nf=2, node_attr_nf=Fa, edge_attr_nf=2, hidden_nf=64, virtual_channels=data["C"], device=dev,
                 n_layers=2, gravity=data["gravity"])
    N, Cc = data["loc_0"].size(0), data["C"]
    a = torch.rand(N, Fa, device=dev) if Fa else None
    flags = L.F_GRAVITY if data["gravity"] is not None else 0
    dims = make_dims(N, N, 0, data["n_graphs"], Cc, 2, flags, data["gravity"], Fa=Fa, node_attr=a)
    named = {k[len("gcl_0."):]: p for k, p in m.named_parameters() if k.startswith("gcl_0.")}
    ptrs = layer_ptrs(named, "")
    grads = {k: torch.zeros_like(p) for k, p in named.items()}
    gptrs = layer_ptrs(grads, "")
    sv = SavedBlock(dims, dev)
    h = torch.randn(N, 64, device=dev)
    G = [torch.randn(N, 64, device=dev) for _ in range(4)] + [torch.randn(N, device=dev) for _ in range(2)]
    gh = torch.zeros(N, 64, device=dev)
    pd, pp, ps, pg = C.byref(dims), C.byref(ptrs), C.byref(sv.c), C.byref(gptrs)

    def call():
        st = torch.cuda.current_stream().cuda_stream
        L.check(L.lib.fegnn_node_pre_forward(pd, pp, L.ptr(h), ps, st))
        L.check(L.lib.fegnn_node_pre_backward(pd, pp, pg, L.ptr(h), *[L.ptr(g) for g in G], L.ptr(gh), st))
    call.keep = (m, a, grads, sv, h, G, gh, dims, ptrs, gptrs)
    return call


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=8, help="alternations of the cases")
    ap.add_argument("--calls", type=int, default=20, help="timed calls per case and round (bench.timed)")
    ap.add_argument("--out", default="profiles/node_attr_cost.json")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # 256 MB > the 126 MB L2
    res = {"card": card(), "what": "ms per call (mean of a block of calls; median / p10 / p90 over the blocks), L2 "
                                  "overwritten before each call, cases alternated block by block in one process; "
                                  "train_step = forward + mse_mmd_loss + backward + FusedAdam (eager, prebuilt CsrGraph); "
                                  "node_pre = fegnn_node_pre_forward + fegnn_node_pre_backward of one layer (default modes)"}
    for name in ("water3d", "water3d_b20"):
        data, hp = bench.make_workload(name, 0, 0)
        cases = {}
        for Fa in WIDTHS:
            cases[f"train_step_Fa{Fa}"] = step_case(data, hp, Fa, dev)
            cases[f"node_pre_Fa{Fa}"] = node_pre_case(data, Fa, dev)
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
