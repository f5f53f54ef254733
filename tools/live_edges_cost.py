#!/usr/bin/env python
"""What a live edge count (FEGNN_F_LIVE_EDGES) costs and what it buys, on the Water-3D shape (8 000 particles, mean degree
~25, C = 3, 4 layers; bench.py's workload and hyperparameters), written to profiles/live_edges_cost.json:

  (a) slack    the captured training step on its exact graph against the same batch on a live graph padded to 1.0x, 1.1x
               and 1.5x its edge count (graph prep inside the step, as bench.py's step has it); every arm its own model,
               optimizer and CUDA graph, the arms alternated in five rounds
  (b) varying  batches of the same node count whose radius graphs differ (jittered positions): today's route (eager step,
               exact CsrGraph.from_radius per batch, two host reads each) against ONE captured step that rebuilds its live
               graph inside (from_radius(capacity=...))
  (c) rollout  a 20-step forward-only rollout that rebuilds the graph from every prediction: eager with the exact
               from_radius against one captured rollout (rebuild_ + forward per step)

Times are CUDA-event times over many steps after warm-up.  The card's name, power limit and max SM clock are read (query
only) in the same run and stored beside the numbers.  A section that fails is recorded as "not measured" with its error.

    python tools/live_edges_cost.py [--out profiles/live_edges_cost.json] [--reps 200]"""
import argparse
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
from fastegnn_b200 import CsrGraph, FastEGNN, FusedAdam, mse_mmd_loss  # noqa: E402

DEV = torch.device("cuda:0")


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def event_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def capture(fn, warm=3):
    """(graph, its output) after `warm` eager calls on a side stream; the output is kept with the graph."""
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


def model_opt(C, gravity):
    torch.manual_seed(0)
    m = FastEGNN(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=64, virtual_channels=C, device=DEV, n_layers=4,
                 gravity=gravity)
    return m, FusedAdam(m.parameters(), lr=5e-4, weight_decay=1e-12)


def train_step(model, opt, t, graph, idx, hp):
    opt.zero_grad(set_to_none=True)
    x, Z = model(node_feat=t["node_feat"], node_loc=t["loc_0"], node_vel=t["vel_0"], edge_index=graph,
                 data_batch=t["batch"], loc_mean=t["loc_mean"])
    loss, _ = mse_mmd_loss(x, t["loc_t"], Z, idx, hp["sigma"], hp["weight"])
    loss.backward()
    opt.step()
    return loss.detach()


def workload():
    data, hp = bench.make_workload("water3d", seed=0, nodes=0)
    C = data["C"]
    idx = bench.sample_indices(data["sizes"], min(hp["sample"] * C, min(data["sizes"])), torch.Generator().manual_seed(0))
    return data, hp, idx.to(DEV)


def spread(v):
    return dict(median=float(np.median(v)), min=float(min(v)), max=float(max(v)))


def slack(reps):
    data, hp, idx = workload()
    C, B = data["C"], data["n_graphs"]
    t = {k: data[k].to(DEV) for k in ("node_feat", "loc_0", "vel_0", "loc_t", "loc_mean", "batch", "edge_index",
                                         "edge_attr")}
    E = int(t["edge_index"].size(1))
    n_live = torch.tensor([E], dtype=torch.int32, device=DEV)
    arms, keep = {}, []
    for f in (None, 1.0, 1.1, 1.5):
        model, opt = model_opt(C, data["gravity"])           # every arm its own model and optimizer state
        if f is None:
            name, step = "exact", (lambda model=model, opt=opt: train_step(
                model, opt, t, CsrGraph(t["edge_index"], t["batch"], t["edge_attr"], B), idx, hp))
        else:
            cap = int(round(f * E))
            ei = torch.cat([t["edge_index"], torch.zeros(2, cap - E, dtype=torch.int64, device=DEV)], dim=1)
            ea = torch.cat([t["edge_attr"], torch.zeros(cap - E, 2, device=DEV)])
            name, step = f"live_{f:.1f}x", (lambda model=model, opt=opt, ei=ei, ea=ea: train_step(
                model, opt, t, CsrGraph(ei, t["batch"], ea, B, n_edges=n_live), idx, hp))
        g, out = capture(step)
        keep.append((model, opt, step, out))
        arms[name] = g
    times = {k: [] for k in arms}
    for _ in range(5):
        for k, g in arms.items():
            times[k].append(event_ms(g.replay, reps))
    return dict(nodes=int(t["loc_0"].size(0)), edges=E, ms_per_step={k: spread(v) for k, v in times.items()})


def varying_batches(n_batches, reps):
    data, hp, idx = workload()
    C, B, N, r = data["C"], data["n_graphs"], int(data["loc_0"].size(0)), data["radius"]
    base = {k: data[k].to(DEV) for k in ("node_feat", "loc_0", "vel_0", "loc_t", "loc_mean", "batch")}
    gen = torch.Generator().manual_seed(1)
    seq = []
    for k in range(n_batches):
        b = dict(base)
        b["loc_0"] = base["loc_0"] + (0.004 * k * torch.randn(N, 3, generator=gen)).to(DEV)
        b["loc_t"] = b["loc_0"] + base["vel_0"]
        seq.append(b)
    Es = [CsrGraph.from_radius(b["loc_0"], b["batch"], B, r, 0.0, 2).E for b in seq]
    cap = int(1.2 * max(Es))
    model, opt = model_opt(C, data["gravity"])
    model_c, opt_c = model_opt(C, data["gravity"])          # the captured arm's own model and optimizer state

    def eager_seq():
        for b in seq:
            train_step(model, opt, b, CsrGraph.from_radius(b["loc_0"], b["batch"], B, r, 0.0, 2), idx, hp)

    static = {k: v.clone() for k, v in seq[0].items()}
    graphs = []

    def live_step():
        g = CsrGraph.from_radius(static["loc_0"], static["batch"], B, r, 0.0, 2, capacity=cap)
        graphs.append(g)
        return train_step(model_c, opt_c, static, g, idx, hp)

    cg, _ = capture(live_step)

    def captured_seq():
        for b in seq:
            static["loc_0"].copy_(b["loc_0"])
            static["loc_t"].copy_(b["loc_t"])
            cg.replay()

    eager_seq()
    captured_seq()
    torch.cuda.synchronize()
    graphs[-1].check()
    te, tc = [], []
    for _ in range(3):
        te.append(event_ms(eager_seq, reps) / n_batches)
        tc.append(event_ms(captured_seq, reps) / n_batches)
    return dict(batches=n_batches, edges=Es, capacity=cap,
                ms_per_step={"eager_exact_from_radius": spread(te), "captured_live": spread(tc)})


def rollout(steps, reps):
    data, hp, _ = workload()
    C, B, r = data["C"], data["n_graphs"], data["radius"]
    t = {k: data[k].to(DEV) for k in ("node_feat", "loc_0", "vel_0", "loc_mean", "batch")}
    model, _ = model_opt(C, data["gravity"])
    model.eval()
    args = dict(node_feat=t["node_feat"], node_vel=t["vel_0"], data_batch=t["batch"], loc_mean=t["loc_mean"])

    @torch.no_grad()
    def eager():
        x = t["loc_0"]
        for _ in range(steps):
            x, _ = model(node_loc=x, edge_index=CsrGraph.from_radius(x, t["batch"], B, r, 0.0, 2), **args)
        return x

    E = CsrGraph.from_radius(t["loc_0"], t["batch"], B, r, 0.0, 2).E
    cap = int(1.5 * E)
    live = CsrGraph.from_radius(t["loc_0"], t["batch"], B, r, 0.0, 2, capacity=cap)
    x_in = t["loc_0"].clone()

    @torch.no_grad()
    def captured_body():
        x = x_in
        for _ in range(steps):
            live.rebuild_(x)
            x, _ = model(node_loc=x, edge_index=live, **args)
        return x

    cg, out = capture(captured_body, warm=1)
    cg.replay()
    want = eager()
    torch.cuda.synchronize()
    live.check()
    te, tc = [], []
    for _ in range(3):
        te.append(event_ms(eager, reps))
        tc.append(event_ms(cg.replay, reps))
    return dict(steps=steps, edges_first_step=E, capacity=cap, max_abs_diff_vs_eager=float((out - want).abs().max()),
                ms_per_rollout={"eager_exact_from_radius": spread(te), "captured_live": spread(tc)})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "live_edges_cost.json"))
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("live_edges_cost.py measures on the GPU; no CUDA device here")
    res = dict(card=card(), card_fields="name, power.limit, clocks.max.sm (nvidia-smi query)")
    for key, fn in (("a_slack", lambda: slack(args.reps)), ("b_varying_batches", lambda: varying_batches(8, 25)),
                    ("c_rollout", lambda: rollout(20, 10))):
        try:
            res[key] = fn()
        except Exception as exc:                   # recorded, not hidden: the section's numbers do not exist
            res[key] = dict(status="not measured", error=f"{type(exc).__name__}: {exc}"[:400],
                            trace=traceback.format_exc()[-1500:])
            break                                  # a device error leaves the context unusable for the next sections
    for key in ("a_slack", "b_varying_batches", "c_rollout"):
        res.setdefault(key, dict(status="not measured"))
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
