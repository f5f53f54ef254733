"""Cost of the deterministic loss kernels: mse_mmd_loss forward + backward with the default kernels and under
torch.use_deterministic_algorithms(True), alternated in one process: bench.timed (CUDA events around each call, L2
overwritten before each call) over blocks of calls, the two modes taking turns block by block.  Writes one JSON file
with the card name and power limit beside the numbers.

    python tools/deterministic_cost.py --out profiles/deterministic_cost.json
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
from fastegnn_b200 import mse_mmd_loss  # noqa: E402

SIGMA, WEIGHT = 1.5, 0.01
# Water-3D (one cloud of 8 000 nodes), water3d_b20 (20 such clouds), config 5 (one graph of 1 M nodes)
SIZES = {"water3d": [8000], "water3d_b20": [8000] * 20, "config5": [1_000_000]}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=10, help="alternations of the two modes")
    ap.add_argument("--calls", type=int, default=20, help="timed calls per mode and round (bench.timed)")
    ap.add_argument("--out", default="profiles/deterministic_cost.json")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # 256 MB > the 126 MB L2
    res = {"card": card(), "what": "mse_mmd_loss forward + backward, ms per call (mean of a block of calls; median / p10 / "
                                  "p90 over the blocks), L2 overwritten before each call"}
    for name, sizes in SIZES.items():
        gen = torch.Generator().manual_seed(0)
        N, B, ns = sum(sizes), len(sizes), 64
        x = torch.randn(N, 3, generator=gen).to(dev).requires_grad_(True)
        tgt = torch.randn(N, 3, generator=gen).to(dev)
        Z = torch.randn(B, 3, 3, generator=gen).to(dev).requires_grad_(True)
        offs = np.concatenate([[0], np.cumsum(sizes)])[:-1]
        idx = torch.stack([torch.randperm(n, generator=gen)[:ns] + int(o) for n, o in zip(sizes, offs)]).to(torch.int32).to(dev)

        def call():
            total, _ = mse_mmd_loss(x, tgt, Z, idx, SIGMA, WEIGHT)
            torch.autograd.grad(total, [x, Z])

        times = {False: [], True: []}
        for r in range(args.rounds + 1):            # round 0 warms both modes up
            for det in (False, True):
                torch.use_deterministic_algorithms(det)
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
        res[name] = dict(nodes=N, graphs=B, **row)
        print(name, json.dumps(row), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
