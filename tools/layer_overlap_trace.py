#!/usr/bin/env python
"""One un-captured Water-3D-size training backward under torch.profiler with fegnn_set_mode("layer_overlap") at 2 and at 0: prints,
per layer, the device time ranges of the virtual backward's heads / trunk kernels and of the edge backward, so that the
overlap of the two branches can be read off (DESIGN.md 3.7).
    python tools/layer_overlap_trace.py [out_dir]      (the Chrome traces go to out_dir, default: the system temp directory)"""
import os
import sys
import tempfile

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tests.gpu_util import make_graph_case  # noqa: E402
from fastegnn_b200 import FastEGNN, _lib  # noqa: E402

out = sys.argv[1] if len(sys.argv) > 1 else tempfile.gettempdir()
os.makedirs(out, exist_ok=True)
dev = "cuda:0"
cfg, params, inp = make_graph_case(3, [8000], 22, 3, L=4, gravity=[0, -1, 0])
m = FastEGNN(node_feat_nf=cfg.node_feat_nf, node_attr_nf=0, edge_attr_nf=cfg.edge_attr_nf, hidden_nf=64,
             virtual_channels=3, device=dev, n_layers=4, gravity=cfg.gravity)
m.load_state_dict({k: v.to(dev) for k, v in params.items()})
t = {k: v.to(dev) for k, v in inp.items()}


def step():
    x0 = t["node_loc"].clone().requires_grad_(True)
    x, Z = m(node_feat=t["node_feat"], node_loc=x0, node_vel=t["node_vel"], edge_index=t["edge_index"],
             data_batch=t["data_batch"], loc_mean=t["loc_mean"], edge_attr=t["edge_attr"])
    ((x * t["wx"]).sum() + (Z * t["wz"]).sum()).backward()


for mode in (2, 0):
    _lib.set_mode("layer_overlap", mode)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    prof.export_chrome_trace(os.path.join(out, f"layer_overlap_{mode}.pt.trace.json"))
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    keys = {"heads": "virtual_bwd_heads", "trunk": "virtual_bwd_trunk", "edge_bwd": "edge_bwd_tc4", "gt": "virtual_bwd_gt"}
    rows = sorted((e.time_range.start, e.time_range.end, k) for e in ev for k, s in keys.items() if s in e.name)
    t0 = rows[0][0] if rows else 0
    print(f"layer_overlap={mode}: kernel, start, end (us from the first listed)")
    for s, e, k in rows:
        print(f"  {k:9s} {s - t0:9.1f} {e - t0:9.1f}  ({e - s:6.1f})")
