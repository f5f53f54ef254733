#!/usr/bin/env python
"""What a differentiable prebuilt graph (CsrGraph.from_radius(..., differentiable=True)) costs, on bench.py's workloads,
written to profiles/graph_grads_cost.json:

  (a) kernel    fegnn_edge_length_backward alone (Fe = 2) on the radius graph of Water-3D (8 000 particles) and of
                water3d_b20 (20 such clouds, one batch)
  (b) eager     bench.py's Water-3D training step (forward, mse_mmd_loss, backward, FusedAdam) on one from_radius graph,
                differentiable off and on (node_loc requires grad in both arms)
  (c) rollout   one captured 3-step rollout training step on Water-3D (each step's own live graph rebuilt from the
                predicted positions, v = (x' - x) / dt) against the workaround without this feature's graph: a live
                from_radius graph for the topology, torch lengths of the padded edge list and CsrGraph(padded,
                n_edges=, differentiable=True), which sorts again every step

Every time is a median of CUDA-event times, L2 overwritten (a 256 MB fill) before each timed call, arms alternated.  The
card's name, power limit and max SM clock are read (query only) in the same run and stored beside the numbers.  A section
that fails is recorded as "not measured" with its error.

    python tools/graph_grads_cost.py [--out profiles/graph_grads_cost.json]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import traceback

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workload generators)
from fastegnn_b200 import CsrGraph, FastEGNN, FusedAdam, _lib, mse_mmd_loss  # noqa: E402
from fastegnn_b200.ops import live_flag, make_dims  # noqa: E402

DEV = torch.device("cuda:0")
FLUSH = None


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def timed(fn):
    """ms of one call, L2 overwritten first."""
    FLUSH.fill_(1)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def alternate(arms, rounds):
    """{name: median ms} of the arms, called in turn `rounds` times after one warm-up call each."""
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(timed(fn))
    return {k: dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v))) for k, v in times.items()}


def workload(name):
    data, hp = bench.make_workload(name, seed=0, nodes=0)
    t = {k: data[k].to(DEV) for k in ("node_feat", "loc_0", "vel_0", "loc_t", "loc_mean", "batch")}
    idx = bench.sample_indices(data["sizes"], min(hp["sample"] * data["C"], min(data["sizes"])),
                               torch.Generator().manual_seed(0)).to(DEV)
    return data, hp, t, idx


def kernel(name, rounds):
    data, _, t, _ = workload(name)
    g = CsrGraph.from_radius(t["loc_0"], t["batch"], data["n_graphs"], data["radius"], 0.0, 2)
    x = t["loc_0"].contiguous()
    g_ea = torch.randn(g.E, 2, device=DEV)
    g_x = torch.zeros(g.N, 3, device=DEV)
    dims = make_dims(g.N, g.N, g.E, g.B, 1, g.Fe, live_flag(g))
    st = torch.cuda.current_stream().cuda_stream

    def call():
        _lib.check(_lib.lib.fegnn_edge_length_backward(C.byref(dims), C.byref(g.c), _lib.ptr(g.rowptr), _lib.ptr(x),
                                                       _lib.ptr(g_ea), _lib.ptr(g_x), st), "fegnn_edge_length_backward")
    res = alternate({"edge_length_backward": call}, rounds)["edge_length_backward"]
    # bytes the kernel has to move at least: rowptr, col, edge_attr[:, 0], g_ea, x of rows and cols, g_x of rows and cols
    nbytes = 4 * (g.N + 1) + 4 * g.E + 4 * g.E + 8 * g.E + 12 * g.N + 12 * g.E + 12 * g.N + 12 * g.E
    return dict(nodes=g.N, edges=g.E, ms=res, min_bytes=nbytes, gbytes_per_s_at_median=nbytes / res["median"] / 1e6)


def model_opt(C_, gravity):
    torch.manual_seed(0)
    m = FastEGNN(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=64, virtual_channels=C_, device=DEV, n_layers=4,
                 gravity=gravity)
    return m, FusedAdam(m.parameters(), lr=5e-4, weight_decay=1e-12)


def eager(rounds):
    data, hp, t, idx = workload("water3d")
    B, r = data["n_graphs"], data["radius"]
    arms = {}
    for diff in (False, True):
        model, opt = model_opt(data["C"], data["gravity"])
        x = t["loc_0"].clone().requires_grad_(True)
        graph = CsrGraph.from_radius(x, t["batch"], B, r, 0.0, 2, differentiable=diff)

        def step(model=model, opt=opt, x=x, graph=graph):
            opt.zero_grad(set_to_none=True)
            xo, Z = model(node_feat=t["node_feat"], node_loc=x, node_vel=t["vel_0"], edge_index=graph, data_batch=t["batch"],
                          loc_mean=t["loc_mean"])
            loss, _ = mse_mmd_loss(xo, t["loc_t"], Z, idx, hp["sigma"], hp["weight"])
            x.grad = None
            loss.backward()
            opt.step()
        arms["differentiable_on" if diff else "differentiable_off"] = step
    return dict(edges=graph.E, ms_per_step=alternate(arms, rounds))


def capture(fn, warm=2):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warm):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    torch.cuda.synchronize()
    return g, out


def rollout(rounds, steps=3, dt=0.5):
    data, hp, t, idx = workload("water3d")
    B, r = data["n_graphs"], data["radius"]
    cap = 2 * CsrGraph.from_radius(t["loc_0"], t["batch"], B, r, 0.0, 2).E       # the predictions move the cloud

    def feature(held, s, x):
        """step s's own differentiable live graph, made on the first call and rebuilt in place afterwards"""
        if len(held) <= s:
            held.append(CsrGraph.from_radius(x, t["batch"], B, r, 0.0, 2, capacity=cap, differentiable=True))
        else:
            held[s].rebuild_(x)
        return held[s]

    def workaround(held, s, x):
        """the topology from a live graph, torch lengths of its padded edge list, and a sorted CsrGraph of both"""
        if len(held) <= s:
            held.append(CsrGraph.from_radius(x, t["batch"], B, r, 0.0, 2, capacity=cap))
        else:
            held[s].rebuild_(x)
        g = held[s]
        live = torch.arange(cap, device=DEV) < g.n_edges
        ei = torch.stack([torch.where(live, g.row[:cap], 0).long(), torch.where(live, g.col[:cap], 0).long()])
        ea = (x[ei[0]] - x[ei[1]]).norm(dim=1, keepdim=True).repeat(1, 2)
        return CsrGraph(ei, t["batch"], ea, B, n_edges=g.n_edges, differentiable=True)

    arms, keep, outs = {}, [], {}
    for name, graph_of in (("differentiable_from_radius", feature), ("torch_lengths_csr_graph_n_edges", workaround)):
        model, opt = model_opt(data["C"], data["gravity"])
        held = []

        def step(model=model, opt=opt, graph_of=graph_of, held=held):
            opt.zero_grad(set_to_none=True)
            x, v, Z = t["loc_0"], t["vel_0"], t["loc_mean"]
            for s in range(steps):
                xo, Z = model(node_feat=t["node_feat"], node_loc=x, node_vel=v, edge_index=graph_of(held, s, x),
                              data_batch=t["batch"], loc_mean=Z)
                x, v = xo, (xo - x) / dt
            loss, _ = mse_mmd_loss(x, t["loc_t"], Z, idx, hp["sigma"], hp["weight"])
            loss.backward()
            opt.step()
            return loss.detach()
        cg, out = capture(step)
        keep.append((model, opt, held))
        arms[name] = cg.replay
        outs[name] = out
    res = alternate(arms, rounds)
    for _, _, held in keep:
        for g in held:
            g.check()
    return dict(steps=steps, capacity=cap, ms_per_step=res, loss_after={k: float(v) for k, v in outs.items()})


def main():
    global FLUSH
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "graph_grads_cost.json"))
    ap.add_argument("--rounds", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("graph_grads_cost.py measures on the GPU; no CUDA device here")
    FLUSH = torch.empty(64 * 1024 * 1024, device=DEV, dtype=torch.float32)
    res = dict(card=card(), card_fields="name, power.limit, clocks.max.sm (nvidia-smi query)")
    sections = (("a_kernel_water3d", lambda: kernel("water3d", 5 * args.rounds)),
                ("a_kernel_water3d_b20", lambda: kernel("water3d_b20", 5 * args.rounds)),
                ("b_eager_step", lambda: eager(args.rounds)),
                ("c_captured_rollout_training_step", lambda: rollout(args.rounds)))
    for key, fn in sections:
        try:
            res[key] = fn()
        except Exception as exc:                   # recorded, not hidden: the section's numbers do not exist
            res[key] = dict(status="not measured", error=f"{type(exc).__name__}: {exc}"[:400],
                            trace=traceback.format_exc()[-1500:])
            break                                  # a device error leaves the context unusable for the next sections
    for key, _ in sections:
        res.setdefault(key, dict(status="not measured"))
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
