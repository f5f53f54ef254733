"""Cost of the deterministic forward-only stack: FastEGNN.forward in eval() under torch.no_grad() (fegnn_model_forward_inference)
with the default kernels and under torch.use_deterministic_algorithms(True), alternated in one process: bench.timed (CUDA
events around each call, L2 overwritten before each call) over blocks of calls, the two modes taking turns block by block.
The graph is built once ahead (CsrGraph.from_radius), so the times are the stack's alone.  Writes one JSON file with the
card name and power limit beside the numbers, and the largest difference between the two modes' outputs.

    python tools/deterministic_inference_cost.py --out profiles/deterministic_inference_cost.json
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from deterministic_cost import card  # noqa: E402
from fastegnn_b200 import CsrGraph, FastEGNN  # noqa: E402

# Water-3D (one cloud of 8 000 nodes), water3d_b20 (20 such clouds), config 5 (one cloud of 1 M nodes, C = 8)
WORKLOADS = {"water3d": (8000, 1, 25.0, 3, [0, -1, 0]), "water3d_b20": (8000, 20, 25.0, 3, [0, -1, 0]),
             "config5": (1_000_000, 1, 30.0, 8, None)}


def inputs(n, B, deg, C, dev):
    clouds = [bench.make_cloud_device(n, deg, C, seed, None, dev) for seed in range(B)]
    cat = lambda k: torch.cat([c[k] for c in clouds]).to(dev)
    batch = torch.cat([torch.full((n,), b, dtype=torch.int64) for b in range(B)]).to(dev)
    loc_mean = torch.cat([c["loc_mean"] for c in clouds]).to(dev)
    graph = CsrGraph.from_radius(cat("loc_0"), batch, B, clouds[0]["radius"], 0.0, 2)
    return dict(node_feat=cat("node_feat"), node_loc=cat("loc_0"), node_vel=cat("vel_0"), edge_index=graph,
                data_batch=batch, loc_mean=loc_mean), graph.E


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=10, help="alternations of the two modes")
    ap.add_argument("--calls", type=int, default=10, help="timed calls per mode and round (bench.timed)")
    ap.add_argument("--only", default=None, help="comma-separated subset of " + ",".join(WORKLOADS))
    ap.add_argument("--out", default="profiles/deterministic_inference_cost.json")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # 256 MB > the 126 MB L2
    res = {"card": card(), "what": "FastEGNN forward-only stack (4 layers, eval + no_grad, graph prebuilt), ms per call "
                                  "(mean of a block of calls; median / p10 / p90 over the blocks), L2 overwritten before "
                                  "each call; max_abs_diff = largest |x_det - x_default| and |Z_det - Z_default|"}
    names = args.only.split(",") if args.only else list(WORKLOADS)
    for name in names:
        n, B, deg, C, gravity = WORKLOADS[name]
        kw, E = inputs(n, B, deg, C, dev)
        torch.manual_seed(0)
        model = FastEGNN(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=64, virtual_channels=C, device=dev,
                         n_layers=4, gravity=gravity).eval()

        def call():
            with torch.no_grad():
                return model(**kw)

        times, outs = {False: [], True: []}, {}
        for r in range(args.rounds + 1):            # round 0 warms both modes up
            for det in (False, True):
                torch.use_deterministic_algorithms(det)
                outs[det] = [t.clone() for t in call()]
                t = bench.timed(call, args.calls, flush)
                if r > 0:
                    times[det].append(t)
        torch.use_deterministic_algorithms(False)
        row = {}
        for det, t in times.items():
            t = np.array(t)
            row["deterministic" if det else "default"] = {"median_ms": float(np.median(t)),
                                                         "p10_ms": float(np.percentile(t, 10)),
                                                         "p90_ms": float(np.percentile(t, 90))}
        row["det_over_default"] = row["deterministic"]["median_ms"] / row["default"]["median_ms"]
        row["max_abs_diff"] = [float((a - b).abs().max()) for a, b in zip(outs[True], outs[False])]
        res[name] = dict(nodes=n * B, graphs=B, edges=int(E), C=C, **row)
        print(name, json.dumps(res[name]), flush=True)
        del model, kw
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
