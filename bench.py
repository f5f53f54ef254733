#!/usr/bin/env python
"""bench.py -- FastEGNN layer path on B200: layer fwd+bwd edges/s and train steps/s.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE
JSON line from rank 0.  A step is one full training step of the reference's loop
(utils/train.py:49-170) on one batch of the workload: 4-layer FastEGNN forward, MSE + weight*MMD,
backward, Adam step.  `value` = (edges x layers processed by all ranks) / (max-over-ranks device time),
inputs resident in HBM; `e2e` = the same with pinned HOST inputs copied in and the loss read back
inside the timed region.

Workloads (BASELINE.json configs):
  water3d   (default, config 4) 8 000 uniform particles, radius graph with mean degree ~25
            (E ~ 2e5 directed edges, ordered by ascending length), C=3, gravity [0,-1,0], B=1.
  water3d_b20  the same clouds batched 20 per step, the reference's training batch (main_simulation.py:46).
  nbody5    (config 1) 100 graphs x 5 particles, 10 edges each: the pure launch-latency regime.
  nbody100  (config 2) 100 graphs x 100 particles, shortest 50% of all ordered pairs.
  protein   (config 3 shape) 50 frames x 855 backbone atoms, 10 A contact graph, shortest 50% kept.
  large     (config 5 shape, scaled by --nodes) uniform cloud, mean degree 30, C=8.
With N>1 ranks: water3d / nbody100 (whole small graphs, as the reference batches them) go one batch per
rank with a single weight-gradient all-reduce per step (--mode dp, SURVEY.md 5.1 mode 1, weak scaling), and
the default line additionally carries a `partitioned` block: ONE config-5 graph (1 M nodes, C=8) spatially
partitioned into N slabs (mode 2; every rank builds its own slab graph on its device), with its 1-GPU time,
the strong-scaling efficiency, the per-layer exchange times and an in-run parity figure against one GPU.
`--workload large` times that partitioned step as the headline instead (strong scaling).
`--mode partitioned` can be forced for water3d too (then 8 000 nodes per rank, weak).

`--impl reference` times the CPU restatement of the reference (oracle/, torch CPU ops in the
reference's op order, all host threads) on the same workload and prints the same line shape.

`--dump-outputs DIR` writes what the last timed (resident) step computed as .npy files, so that two builds run with the
same arguments, hence on the same seeded inputs, can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

H, LAYERS = 64, 4


# ----------------------------------------------------------------------------- workloads
def radius_graph_np(pts: np.ndarray, r: float):
    from scipy.spatial import cKDTree
    pairs = cKDTree(pts).query_pairs(r, output_type="ndarray")           # i < j
    row = np.concatenate([pairs[:, 0], pairs[:, 1]])
    col = np.concatenate([pairs[:, 1], pairs[:, 0]])
    return row, col


def make_cloud(n: int, mean_deg: float, C: int, seed: int, gravity, r: float = 0.035, vel_std: float = 0.01):
    """Uniform points in a cube sized so that radius r gives `mean_deg` neighbours
    (datasets/simulation/dataset.py:80); edges ordered by ascending length like cutoff_edge (:96-101)."""
    rng = np.random.default_rng(seed)
    rho = mean_deg / (4.0 / 3.0 * math.pi * r ** 3)
    side = (n / rho) ** (1.0 / 3.0)
    x = (rng.random((n, 3)) * side).astype(np.float32)
    row, col = radius_graph_np(x.astype(np.float64), r)
    length = np.linalg.norm(x[row] - x[col], axis=1)
    order = np.argsort(length, kind="stable")
    row, col, length = row[order], col[order], length[order].astype(np.float32)
    v = (rng.standard_normal((n, 3)) * vel_std).astype(np.float32)
    q = rng.choice([-1.0, 1.0], size=n).astype(np.float32)
    node_feat = np.stack([np.linalg.norm(v, axis=1), q / np.abs(q).max()], axis=1).astype(np.float32)
    loc_t = (x + v + rng.standard_normal((n, 3)).astype(np.float32) * 1e-3).astype(np.float32)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    return dict(node_feat=t(node_feat), loc_0=t(x), vel_0=t(v), loc_t=t(loc_t),
                edge_index=t(np.stack([row, col]).astype(np.int64)),
                edge_attr=t(np.stack([length, length], axis=1)),                 # utils/train.py:41-43
                batch=torch.zeros(n, dtype=torch.int64),
                loc_mean=t(x.mean(0, keepdims=True).T[None].repeat(C, axis=2).astype(np.float32)),
                n_graphs=1, C=C, gravity=gravity, sizes=[n], radius=r)


def make_cloud_batch(n: int, B: int, mean_deg: float, C: int, seed: int, gravity):
    """B independent clouds batched the way the reference's DataLoader collates them (main_simulation.py:46 trains with
    batch_size 20): node tensors concatenated, edge_index offset by the cumulative node count."""
    parts = [make_cloud(n, mean_deg, C, seed * 1000 + b, gravity) for b in range(B)]
    cat = lambda k: torch.cat([p[k] for p in parts])
    ei = torch.cat([p["edge_index"] + b * n for b, p in enumerate(parts)], dim=1)
    return dict(node_feat=cat("node_feat"), loc_0=cat("loc_0"), vel_0=cat("vel_0"), loc_t=cat("loc_t"), edge_index=ei,
                edge_attr=cat("edge_attr"), batch=torch.arange(B).repeat_interleave(n), loc_mean=cat("loc_mean"),
                n_graphs=B, C=C, gravity=gravity, sizes=[n] * B, radius=parts[0]["radius"])


def make_protein(n: int, B: int, cutoff_rate: float, C: int, seed: int, r: float = 10.0, blob_sigma: float = 9.5):
    """Config 3 shape (datasets/protein/dataset.py:89,146-156,208-213): B frames of n backbone atoms as a compact blob
    (the AdK trajectory is not available offline; sigma chosen so that ~3.4e4 directed edges per frame survive, the
    middle of SURVEY.md 8's 2-5e4 estimate), 10 A contact graph without self loops, shortest (1 - cutoff_rate)
    of the edges kept, ordered by ascending length."""
    rng = np.random.default_rng(seed)
    parts = []
    for b in range(B):
        x = (rng.standard_normal((n, 3)) * blob_sigma).astype(np.float32)
        row, col = radius_graph_np(x.astype(np.float64), r)
        length = np.linalg.norm(x[row] - x[col], axis=1)
        order = np.argsort(length, kind="stable")[:int(row.size * (1 - cutoff_rate))]
        row, col, length = row[order], col[order], length[order].astype(np.float32)
        v = (rng.standard_normal((n, 3)) * 0.1).astype(np.float32)
        q = rng.random(n).astype(np.float32)
        parts.append(dict(x=x, v=v, nf=np.stack([np.linalg.norm(v, axis=1), q / q.max()], 1).astype(np.float32),
                          ei=np.stack([row, col]).astype(np.int64) + b * n, ea=np.stack([length, length], 1),
                          lm=x.mean(0, keepdims=True).T.repeat(C, axis=1)))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    cat = lambda k, ax=0: np.concatenate([p[k] for p in parts], axis=ax)
    x, v = cat("x"), cat("v")
    return dict(node_feat=t(cat("nf")), loc_0=t(x), vel_0=t(v), loc_t=t((x + v).astype(np.float32)),
                edge_index=t(cat("ei", 1)), edge_attr=t(cat("ea").astype(np.float32)),
                batch=torch.arange(B).repeat_interleave(n), loc_mean=t(np.stack([p["lm"] for p in parts]).astype(np.float32)),
                n_graphs=B, C=C, gravity=None, sizes=[n] * B)


def make_nbody(n: int, B: int, cutoff: float, C: int, seed: int):
    """datagen/system.py:21-39 initial conditions + datasets/nbody/dataset.py:102-113 edge selection."""
    rng = np.random.default_rng(seed)
    sigma = (n / 5.0) ** (1.0 / 3.0) + 0.1
    xs, vs, nfs, rows, cols, eas, lms = [], [], [], [], [], [], []
    keep = int(n * (n - 1) * (1 - cutoff))
    for b in range(B):
        x = (rng.standard_normal((n, 3)) * sigma).astype(np.float32)
        v = rng.standard_normal((n, 3)).astype(np.float32)
        v = (v / np.linalg.norm(v, axis=1, keepdims=True) * 0.5).astype(np.float32)
        q = rng.choice([-1.0, 1.0], size=n).astype(np.float32)
        d = np.linalg.norm(x[:, None] - x[None], axis=2)
        np.fill_diagonal(d, 1e18)
        idx = np.argsort(d.reshape(-1), kind="stable")[:keep]
        r, c = idx // n, idx % n
        ln = d.reshape(-1)[idx].astype(np.float32)
        xs.append(x); vs.append(v); nfs.append(np.stack([np.linalg.norm(v, axis=1), q], 1).astype(np.float32))
        rows.append(r + b * n); cols.append(c + b * n); eas.append(np.stack([ln, ln], 1))
        lms.append(x.mean(0, keepdims=True).T.repeat(C, axis=1))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    x = np.concatenate(xs)
    v = np.concatenate(vs)
    return dict(node_feat=t(np.concatenate(nfs)), loc_0=t(x), vel_0=t(v), loc_t=t((x + v).astype(np.float32)),
                edge_index=t(np.stack([np.concatenate(rows), np.concatenate(cols)]).astype(np.int64)),
                edge_attr=t(np.concatenate(eas).astype(np.float32)),
                batch=torch.arange(B).repeat_interleave(n), loc_mean=t(np.stack(lms).astype(np.float32)),
                n_graphs=B, C=C, gravity=None, sizes=[n] * B)


def make_workload(name: str, seed: int, nodes: int):
    if name == "water3d":
        return make_cloud(nodes or 8000, 25.0, 3, seed, [0, -1, 0]), dict(sigma=1.0, weight=0.01, sample=3)
    if name == "water3d_b20":
        return make_cloud_batch(nodes or 8000, 20, 25.0, 3, seed, [0, -1, 0]), dict(sigma=1.0, weight=0.01, sample=3)
    if name == "nbody5":      # config 1: datagen default --n_isolated 5, batch 100 (main_nbody.py:46), 10 edges per graph
        return make_nbody(5, 100, 0.5, 3, seed), dict(sigma=1.5, weight=0.01, sample=3)
    if name == "nbody100":
        return make_nbody(100, 100, 0.5, 3, seed), dict(sigma=1.5, weight=0.01, sample=3)
    if name == "protein":
        return make_protein(855, 50, 0.5, 3, seed), dict(sigma=1.5, weight=0.01, sample=3)
    if name == "large":
        return make_cloud(nodes or 1_000_000, 30.0, 8, seed, None), dict(sigma=1.0, weight=0.01, sample=3)
    raise SystemExit(f"unknown workload {name}")


def sample_indices(sizes, ns, gen):
    """Global node indices of the reference's per-graph torch.randperm(n_b)[:ns] (utils/train.py:131,152)."""
    out, off = [], 0
    for n in sizes:
        out.append(torch.randperm(n, generator=gen)[:ns] + off)
        off += n
    return torch.stack(out).to(torch.int32)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            p = [s.strip() for s in ln.split(",")]
            if len(p) < 6 or not p[0].isdigit():
                continue
            sm.append(int(p[0])); mx = int(p[1])
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=mx, reasons=sorted(reasons),
                    samples=len(sm))


# ----------------------------------------------------------------------------- reference arm (CPU)
def oracle_step_fn(data, hp, device="cpu", model="fastegnn"):
    """The reference's training step (utils/train.py:49-170) on the restatement of the model in the reference's own
    torch op chain; device="cuda" gives the eager-PyTorch-on-the-same-GPU bar (--gpu-eager-bar)."""
    from oracle import fastegnn_oracle as orc
    cfg = orc.OracleConfig(node_feat_nf=2, edge_attr_nf=2, hidden_nf=H, virtual_channels=data["C"], n_layers=LAYERS,
                           gravity=data["gravity"])
    if model == "fastrf":
        from oracle import fastrf_oracle as rfo
        make_params, forward = rfo.make_params, rfo.fastrf_forward
    else:
        make_params, forward = orc.make_params, orc.fastegnn_forward
    params = {k: v.clone().to(device).requires_grad_(True) for k, v in make_params(cfg, 0).items()}
    if device != "cpu":
        data = {k: (v.to(device) if isinstance(v, torch.Tensor) else v) for k, v in data.items()}
    opt = torch.optim.Adam(list(params.values()), lr=5e-4, weight_decay=1e-12)
    gen = torch.Generator().manual_seed(0)
    ns = min(hp["sample"] * data["C"], min(data["sizes"]))
    offs = np.concatenate([[0], np.cumsum(data["sizes"])[:-1]])

    def step():
        opt.zero_grad()
        x, Z = forward(params, cfg, data["node_feat"], data["loc_0"], data["vel_0"], data["edge_index"],
                       data["batch"], data["loc_mean"], data["edge_attr"])
        loss = torch.nn.functional.mse_loss(x, data["loc_t"])
        idx = sample_indices(data["sizes"], ns, gen).long()
        local = [(idx[b] - int(offs[b])).to(device) for b in range(len(data["sizes"]))]
        loss = loss + hp["weight"] * orc.mmd_loss(x, Z, data["batch"], hp["sigma"], local)
        loss.backward()
        opt.step()
        return float(loss.detach())
    return step


def time_cpu(step, warmup, steps):
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    return sum(ts) / len(ts)


# ----------------------------------------------------------------------------- the timed step
DTYPE_DEFAULT = ("tf32: tcgen05 TF32 operand tiles with fp32 accumulation and tanh.approx SiLU in the edge and virtual "
                 "phases (fp16 operands with power-of-two scales in the edge backward), TF32 tiles in the node-side backward, "
                 "error-compensated 3xTF32 tiles (fp32-grade) in the node-side forward, fp32 FMA in the per-graph phases "
                 "(the reference is strict fp32; the fp32-kernel figure is in `fp32_mode`)")


def make_cloud_device(n: int, mean_deg: float, C: int, seed: int, gravity, dev, r: float = 0.035, vel_std: float = 0.01):
    """make_cloud for clouds whose graph is built ON THE DEVICE (fegnn_radius_graph_*, SURVEY.md 8 f2): same point / velocity
    / feature recipe, no KD-tree and no host edge list (3e7 edges at config 5).  Returns host tensors + the radius."""
    rng = np.random.default_rng(seed)
    rho = mean_deg / (4.0 / 3.0 * math.pi * r ** 3)
    side = (n / rho) ** (1.0 / 3.0)
    x = (rng.random((n, 3)) * side).astype(np.float32)
    v = (rng.standard_normal((n, 3)) * vel_std).astype(np.float32)
    q = rng.choice([-1.0, 1.0], size=n).astype(np.float32)
    node_feat = np.stack([np.linalg.norm(v, axis=1), q], axis=1).astype(np.float32)
    loc_t = (x + v + rng.standard_normal((n, 3)).astype(np.float32) * 1e-3).astype(np.float32)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    return dict(node_feat=t(node_feat), loc_0=t(x), vel_0=t(v), loc_t=t(loc_t), batch=torch.zeros(n, dtype=torch.int64),
                loc_mean=t(x.mean(0, keepdims=True).T[None].repeat(C, axis=2).astype(np.float32)),
                n_graphs=1, C=C, gravity=gravity, sizes=[n], radius=r)


class StepBench:
    """One workload's training step (utils/train.py:49-170: forward, MSE + weight * MMD, backward, optimizer step) on this
    rank, captured as ONE CUDA graph when possible; `resident()` replays it on inputs already in HBM, `e2e()` first copies
    every input from pinned host memory and reads the loss back.

    mode "single": one rank or whole graphs per rank (+ weight-gradient all-reduce when world > 1).
    mode "partitioned": `runner` (PartitionedFastEGNN) drives this rank's slab of one graph."""

    def __init__(self, data, hp, dev, world=1, rank=0, model_name="fastegnn", graph=None, runner_factory=None,
                 use_cuda_graph=True, n_global=None, idx_all=None, mmd_scales=(1.0, 1.0), seed=0):
        import torch.distributed as dist
        from fastegnn_b200 import FastEGNN, FusedAdam, _lib, mmd_loss, mse_mmd_loss
        self._lib, self.dev, self.world, self.hp = _lib, dev, world, hp
        C = data["C"]
        torch.manual_seed(seed)
        if model_name == "fastrf":
            from fastegnn_b200 import FastRF as Model
        else:
            Model = FastEGNN
        self.model = model = Model(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=H, virtual_channels=C, device=dev,
                                   n_layers=LAYERS, gravity=data["gravity"])
        self.opt = opt = FusedAdam(model.parameters(), lr=5e-4, weight_decay=1e-12)   # torch.optim.Adam's step, one launch
        params = [p for p in model.parameters()]
        self.runner = runner = runner_factory(model) if runner_factory is not None else None
        part = runner is not None
        prebuilt = graph is not None or part and data.get("edge_index") is None
        keys = ["node_feat", "loc_0", "vel_0", "loc_t", "loc_mean"] + ([] if part else ["batch"]) + \
               ([] if prebuilt else ["edge_index", "edge_attr"])
        self.keys = keys
        if idx_all is None:
            gen = torch.Generator().manual_seed(0)
            ns = min(hp["sample"] * C, min(data["sizes"]))
            idx_all = sample_indices(data["sizes"], ns, gen)                    # [B, ns] global node ids
        self.host = host = {k: data[k].pin_memory() for k in keys}
        self.dev_in = dev_in = {k: host[k].to(dev) for k in keys}
        self.idx_host = idx_all.pin_memory()
        self.idx_dev = self.idx_host.to(dev)
        n_own = runner.comm.N if part else int(data["loc_0"].size(0))
        n_glob = n_global if n_global is not None else n_own
        svv, srv = mmd_scales

        def allreduce_grads():
            flat = opt.flat_grad() if hasattr(opt, "flat_grad") else None
            if flat is not None:                 # the gradients ARE one flat buffer: all-reduce it in place
                dist.all_reduce(flat)
                flat.div_(world)
                return
            grads = [p.grad for p in params if p.grad is not None]
            flat = torch._utils._flatten_dense_tensors(grads)
            dist.all_reduce(flat)
            flat.div_(world)
            torch._foreach_copy_(grads, list(torch._utils._unflatten_dense_tensors(flat, grads)))

        def train_step(t, idx):
            opt.zero_grad(set_to_none=True)
            if part:
                x, Z = runner(t["node_feat"], t["loc_0"], t["vel_0"], graph if prebuilt else t["edge_index"],
                              t["loc_mean"], None if prebuilt else t["edge_attr"], n_global=n_glob)
                # MSE over ALL nodes and the MMD term, written as a sum of rank-local shares
                loss = ((x - t["loc_t"][:n_own]) ** 2).sum() / (3.0 * n_glob) + \
                    hp["weight"] * mmd_loss(x, Z, idx, hp["sigma"], svv, srv)
                loss.backward()
                runner.allreduce_gradients()
            else:
                x, Z = model(node_feat=t["node_feat"], node_loc=t["loc_0"], node_vel=t["vel_0"],
                             edge_index=graph if prebuilt else t["edge_index"], data_batch=t["batch"],
                             loc_mean=t["loc_mean"], edge_attr=None if prebuilt else t["edge_attr"])
                # utils/train.py:104-163: MSE + weight * MMD -- one launch per direction (mse_mmd_loss), not ten torch kernels
                loss, mse = mse_mmd_loss(x, t["loc_t"], Z, idx, hp["sigma"], hp["weight"])
                loss.backward()
                if world > 1:
                    allreduce_grads()
            opt.step()
            # what the step hands its caller (--dump-outputs): detached views, so no autograd state outlives the step;
            # a captured graph's replays rewrite these same tensors
            self.outputs = dict(node_loc=x.detach(), virtual_node_loc=Z.detach(), loss=loss.detach())
            if not part:
                self.outputs["mse"] = mse.detach()
            return loss
        self.train_step = train_step
        # ---- the whole step (graph prep, 4-layer fwd, losses, bwd, collectives, Adam) as ONE CUDA graph:
        #      the C ABI never allocates or synchronises, so every launch of a step is capturable.
        self.g, self.loss, self.why, self.per_step, self.pipe = None, None, None, None, None
        if use_cuda_graph:
            try:
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for _ in range(3):
                        train_step(dev_in, self.idx_dev)
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                c0 = _lib.lib.fegnn_launch_count()
                with torch.cuda.graph(g):
                    self.loss = train_step(dev_in, self.idx_dev)
                self.per_step = int(_lib.lib.fegnn_launch_count() - c0)     # kernels of this library in the graph
                self.g = g
            except Exception as exc:                                      # pragma: no cover - reported in the JSON line
                self.g, self.why = None, f"{type(exc).__name__}: {exc}"[:300]
                torch.cuda.synchronize()

    def resident(self):
        if self.g is not None:
            self.g.replay()
            return self.loss
        return self.train_step(self.dev_in, self.idx_dev)

    def e2e_pipelined(self):
        """End to end through fastegnn_b200.PipelinedStep: the pinned-host inputs of step k+1 travel on a copy stream
        while step k computes (double-buffered device inputs, two captured graphs); the loss is read back every step."""
        if self.pipe is None:
            from fastegnn_b200 import PipelinedStep
            host = dict(self.host, idx=self.idx_host)
            self.pipe = PipelinedStep(lambda t: self.train_step(t, t["idx"]), host, self.dev)
            self.pipe_host = host
            self.pipe.prefetch(host)
        return self.pipe.run_and_read(self.pipe_host)

    def e2e(self):
        if self.g is not None:
            for k in self.keys:                                           # pinned host -> the graph's static inputs
                self.dev_in[k].copy_(self.host[k], non_blocking=True)
            self.idx_dev.copy_(self.idx_host, non_blocking=True)
            self.g.replay()
            return self.loss.item()                                       # device->host read of the loss
        t = {k: self.host[k].to(self.dev, non_blocking=True) for k in self.keys}
        idx = self.idx_host.to(self.dev, non_blocking=True)
        return self.train_step(t, idx).item()

    def h2d_bytes(self):
        return sum(self.host[k].numel() * self.host[k].element_size() for k in self.keys) + self.idx_host.numel() * 4

    def launches(self, steps, measured):
        return self.per_step * steps if self.g is not None else measured


def timed(fn, steps, flush):
    """Per-step CUDA events on the launching (current) stream, L2 flushed before each step."""
    evs = []
    for _ in range(steps):
        flush.fill_(1)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        evs.append((s, e))
    torch.cuda.synchronize()
    return sum(s.elapsed_time(e) for s, e in evs) / steps     # ms


DUMP_ARRAY_BYTES = 16_000_000        # per array; at most four arrays can reach it, so a dump stays under 64 MB


def dump_outputs(sb, out_dir):
    """Write what the last step of `sb` handed its caller to out_dir/<name>.npy (float32): node_loc [N,3],
    virtual_node_loc [B,3,C], loss (and mse) [1], the parameters after the optimizer step and the gradients it applied
    (params / grads: flat, in model.parameters() order, zeros where a parameter got no gradient).  An array above
    DUMP_ARRAY_BYTES keeps a fixed sample of its rows: sorted row ids drawn with numpy seed 0 from the row count alone, the
    same in every run of the same arguments."""
    params = list(sb.model.parameters())
    arrays = dict(sb.outputs)
    arrays["params"] = torch.cat([p.detach().reshape(-1) for p in params])
    arrays["grads"] = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).detach().reshape(-1)
                                 for p in params])
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.float().cpu().numpy().reshape(t.shape if t.dim() else (1,))
        row_bytes = a[:1].nbytes
        if a.nbytes > DUMP_ARRAY_BYTES:
            k = DUMP_ARRAY_BYTES // row_bytes
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], k, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a))


def quick_config(name, dev, flush, steps=5, warmup=3):
    """One line of the per-config table (BASELINE.json configs 1-5 on ONE GPU): ms per training step, resident."""
    if name == "large":
        data, hp = make_cloud_device(1_000_000, 30.0, 8, 0, None, dev), dict(sigma=1.0, weight=0.01, sample=3)
        from fastegnn_b200 import CsrGraph
        graph = CsrGraph.from_radius(data["loc_0"].to(dev), data["batch"].to(dev), 1, data["radius"], 0.0, 2)
        E = graph.E
        note = "graph built on the device once (fegnn_radius_graph_*), CSR reused by every step"
    else:
        data, hp = make_workload(name, seed=0, nodes=0)
        graph, E, note = None, int(data["edge_index"].size(1)), "edge_index re-sorted to CSR inside every step"
    sb = StepBench(data, hp, dev, graph=graph)
    for _ in range(warmup):
        sb.resident()
    ms = timed(sb.resident, steps, flush)
    out = dict(nodes=int(data["loc_0"].size(0)), edges=int(E), graphs=data["n_graphs"], C=data["C"], ms_per_step=round(ms, 4),
               layer_edges_per_s=E * LAYERS / (ms * 1e-3), cuda_graph=sb.g is not None, graph=note)
    del sb, graph, data
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="water3d", choices=["water3d", "water3d_b20", "nbody5", "nbody100", "protein", "large"])
    ap.add_argument("--model", default="fastegnn", choices=["fastegnn", "fastrf"],
                    help="fastrf: the radial-field sibling (models/FastRF.py, main_protein.py:114) on the same kernels")
    ap.add_argument("--nodes", type=int, default=0)
    ap.add_argument("--mode", default="auto", choices=["auto", "dp", "partitioned"])
    ap.add_argument("--halo", default="fused", choices=["fused", "p2p", "nccl"],
                    help="partitioned path: fused payload+signal kernels over peer memory (default), peer-memory kernels + "
                         "symmetric-memory barrier, or NCCL all-to-all")
    ap.add_argument("--no-graph", action="store_true", help="do not capture the training step in a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-phases", action="store_true")
    ap.add_argument("--no-gpu-eager-bar", action="store_true",
                    help="skip timing the reference's torch op chain (oracle/ restatement) eagerly on the same GPU")
    ap.add_argument("--no-per-config", action="store_true", help="skip the per-config table (configs 1-5, one GPU)")
    ap.add_argument("--no-fp32-line", action="store_true", help="skip the fp32-kernel timing of the same step")
    ap.add_argument("--no-partitioned-block", action="store_true",
                    help="N > 1, default workload: skip the partitioned config-5 block (1 M nodes in N slabs)")
    ap.add_argument("--part-nodes", type=int, default=1_000_000, help="nodes of the partitioned block's graph")
    ap.add_argument("--rollout", action="store_true", help="also time the forward-only rollout mode (utils/train.py:191)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs; "
                         "with several ranks, rank 0's share)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm's step")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert args.warmup >= 3 or args.impl == "reference", "timing rules: at least 3 warm-up steps"

    mode = args.mode
    if mode == "auto":
        # small / batched graphs (configs 1-4) go whole to the ranks; one big graph (config 5) is partitioned
        mode = "partitioned" if world > 1 and args.impl == "b200" and args.workload == "large" else "dp"
    part = mode == "partitioned" and world > 1
    device_graph = args.workload == "large" and args.impl == "b200"       # graph built on the device, never on the host
    if device_graph:
        data, hp = make_cloud_device(args.nodes or 1_000_000, 30.0, 8, 0 if part else rank, None, None), \
            dict(sigma=1.0, weight=0.01, sample=3)
    elif part:
        nodes = args.nodes or (8000 * world if args.workload == "water3d" else 0)
        data, hp = make_workload(args.workload, seed=0, nodes=nodes)          # every rank builds the same global graph
    else:
        data, hp = make_workload(args.workload, seed=rank, nodes=args.nodes)
    N, B, C = int(data["loc_0"].size(0)), data["n_graphs"], data["C"]
    E = int(data["edge_index"].size(1)) if "edge_index" in data else None   # device-built graphs: known after the build
    scaling = "weak" if not (part and args.workload == "large") else "strong"
    metric = "layer fwd+bwd edges/sec (full train step: fwd+MSE+MMD+bwd+Adam), Water-3D shape"
    cores = os.cpu_count() or 1

    def make_config(E_, par):
        return dict(workload=f"{args.workload}: N={N} nodes, E={E_} directed edges{' (global)' if part else ''}, "
                             f"B={B} graph(s), C={C}, L={LAYERS}, H={H}, gravity={data['gravity']}"
                             f"{', model=FastRF' if args.model == 'fastrf' else ''}; "
                             f"step = fwd + MSE + {hp['weight']}*MMD + bwd + Adam",
                    l2="flushed (256 MiB write) before every timed step", parallelism=par)

    if args.impl == "reference":
        if rank != 0:
            return
        torch.set_num_threads(cores)
        step = oracle_step_fn(data, hp, model=args.model)
        w, k = args.warmup, args.steps
        t = time_cpu(step, w, k)
        val = E * LAYERS / t
        line = dict(impl="reference", metric=metric, value=val, unit="edges/s", n_gpus=args.gpus,
                    steps=k, warmup=w, ms_per_step=t * 1e3,
                    steps_per_sec=1.0 / t, higher_is_better=True, scaling=scaling, vs_baseline=None,
                    dtype="f32 (torch CPU ops)", data="synthetic", config=make_config(E, "1 rank"),
                    cpu_baseline=dict(value=val, unit="edges/s", cores=cores, kind="port",
                                      sample="the full workload, one training step per timed step: oracle/ restates the "
                                             "reference's torch op chain and is pinned bit-for-bit to golden vectors of "
                                             "the unmodified reference; /root/reference itself does not exist on the GPU "
                                             "box, so the port is what can be timed there"),
                    e2e=dict(value=val, unit="edges/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------ B200 arm
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"         # keep stdout to the one JSON line (NCCL prints its banner there)
        dist.init_process_group("nccl", device_id=dev)
    from fastegnn_b200 import _lib

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    par = "1 rank"
    graph, runner_factory, idx_all, scales, halo_used = None, None, None, (1.0, 1.0), None
    bench_data = data
    if part:
        bench_data, graph, runner_factory, idx_all, scales, halo_used, E = partition_setup(
            data, hp, args, world, rank, dev, device_graph)
    elif device_graph:
        from fastegnn_b200 import CsrGraph
        graph = CsrGraph.from_radius(data["loc_0"].to(dev), data["batch"].to(dev), 1, data["radius"], 0.0, 2)
        E = graph.E
    if world > 1:
        par = (f"{world} ranks, ONE graph in {world} slabs built per rank on its device: halo exchange ({halo_used}) + "
               "per-graph all-reduce per layer, weight-gradient all-reduce per step") if part else \
              f"{world} ranks, whole graphs per rank, weight-gradient all-reduce per step"
    config = make_config(E, par)
    sb = StepBench(bench_data, hp, dev, world=world, rank=rank, model_name=args.model, graph=graph,
                   runner_factory=runner_factory, use_cuda_graph=not args.no_graph, n_global=N, idx_all=idx_all,
                   mmd_scales=scales)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        sb.resident()
        sb.e2e()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = _lib.lib.fegnn_launch_count()
    barrier()
    ms = timed(sb.resident, args.steps, flush)
    barrier()
    launches = sb.launches(args.steps, _lib.lib.fegnn_launch_count() - launches0)
    if args.dump_outputs and rank == 0:
        dump_outputs(sb, args.dump_outputs)
    ms_e2e_serial = timed(sb.e2e, args.steps, flush)
    barrier()
    pipelined = not part and not args.no_graph
    if pipelined:
        for _ in range(args.warmup):
            sb.e2e_pipelined()
        barrier()
        ms_e2e = timed(sb.e2e_pipelined, args.steps, flush)
        if sb.pipe.graphs[0] is None:
            pipelined = False
    else:
        ms_e2e = ms_e2e_serial
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        tt = torch.tensor([ms, ms_e2e, ms_e2e_serial], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_e2e_serial = float(tt[2])
        ee = torch.tensor([E], device=dev, dtype=torch.float64)
        dist.all_reduce(ee)
        ms, ms_e2e, E_all = float(tt[0]), float(tt[1]), float(ee[0])    # partitioned: E is this rank's share of the edges
    else:
        E_all = float(E)
    if part and hasattr(sb.runner.comm, "check"):
        sb.runner.comm.check()

    line = None
    if rank == 0:
        line = dict(metric=metric, value=E_all * LAYERS / (ms * 1e-3), unit="edges/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms, steps_per_sec=1e3 / ms, higher_is_better=True, scaling=scaling,
                    vs_baseline=None, dtype=DTYPE_DEFAULT if _lib.get_mode("edge_forward") else "f32 (fp32 FMA kernels)",
                    data="synthetic", config=config, clocks=clocks,
                    e2e=dict(value=E_all * LAYERS / (ms_e2e * 1e-3), unit="edges/s", ms_per_step=ms_e2e,
                             h2d_bytes_per_step=sb.h2d_bytes(), d2h_bytes_per_step=4,
                             ms_per_step_serial_copy=ms_e2e_serial,
                             how=("fastegnn_b200.PipelinedStep: every step copies its batch from pinned host memory and reads "
                                  "the loss back; the copy of step k+1's inputs runs on a copy stream while step k computes "
                                  "(double-buffered device inputs, one captured graph per set) -- all copies lie inside the "
                                  "timed region; ms_per_step_serial_copy is the same with the copy in front of the step on "
                                  "the compute stream") if pipelined else
                                 "pinned host -> device copy of every input on the compute stream, then the step, then the "
                                 "loss read-back"),
                    gpu_launches=int(launches), cuda_graph=sb.g is not None,
                    modes={ph: _lib.get_mode(ph) for ph in _lib.PHASES})
        if part:
            line["config"]["workload"] = line["config"]["workload"].replace(f"E={E} ", f"E={int(E_all)} ")
        if sb.why:
            line["cuda_graph_error"] = sb.why
        if args.model != "fastegnn":
            line["model"] = args.model
        if world == 1 and not part:
            single_gpu_extras(line, args, sb, data, hp, dev, flush, E, N, B, C, cores)
    if world > 1 and not part and args.workload == "water3d" and not args.no_partitioned_block:
        # north_star item 5 in the driver's scaling record: ONE config-5 graph partitioned over the N ranks
        del sb
        torch.cuda.empty_cache()
        try:
            blk = partitioned_block(args, world, rank, dev, flush)
        except Exception as exc:                                   # reported, never hides the headline numbers
            blk = dict(error=f"{type(exc).__name__}: {exc}"[:400])
        if rank == 0:
            line["partitioned"] = blk
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        # a captured graph still references the communicator: skip the (occasionally hanging) NCCL teardown
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)


def single_gpu_extras(line, args, sb, data, hp, dev, flush, E, N, B, C, cores):
    """Rank-0, one-GPU additions to the line: per-phase times + roofline (against measured probes), the fp32-kernel
    figure of the same step, the graph build, the per-config table, the CPU port and the eager-PyTorch-on-this-GPU bar."""
    from fastegnn_b200 import _lib
    has_edges = "edge_index" in data
    if not args.no_phases and args.model == "fastegnn" and has_edges:
        line.update(phase_profile(sb.model, sb.dev_in, dev, data, E, N, B, C, flush))
        if data.get("radius") is not None:
            try:
                line["graph_build"] = graph_build_profile(data, sb.dev_in, dev, B, flush)
            except Exception as exc:                          # reported, never hides the headline numbers
                line["graph_build"] = dict(error=f"{type(exc).__name__}: {exc}"[:300])
    if not args.no_fp32_line and has_edges:
        old = {ph: _lib.get_mode(ph) for ph in _lib.PHASES}
        try:
            _lib.set_precision("fp32")
            sb32 = StepBench(data, hp, dev, model_name=args.model, use_cuda_graph=not args.no_graph)
            for _ in range(3):
                sb32.resident()
            ms32 = timed(sb32.resident, max(5, min(args.steps, 20)), flush)
            line["fp32_mode"] = dict(ms_per_step=ms32, value=E * LAYERS / (ms32 * 1e-3), unit="edges/s",
                                     what="the same step with every phase on the fp32 FMA kernels "
                                          "(FEGNN_PRECISION=fp32: parity with the fp32 reference at 2e-6 / 8e-5)")
            del sb32
        except Exception as exc:
            line["fp32_mode"] = dict(error=f"{type(exc).__name__}: {exc}"[:300])
        finally:
            for ph, m in old.items():
                _lib.set_mode(ph, m)
    if has_edges:
        try:
            line["rollout"] = rollout_profile(sb.model, sb.dev_in, dev, E, flush)
        except Exception as exc:
            line["rollout"] = dict(error=f"{type(exc).__name__}: {exc}"[:300])
    if not args.no_per_config and args.workload == "water3d" and not args.nodes:
        table = {"water3d (config 4)": dict(nodes=N, edges=E, graphs=B, C=C, ms_per_step=round(line["ms_per_step"], 4),
                                            layer_edges_per_s=line["value"], cuda_graph=line["cuda_graph"])}
        for name, tag in (("nbody5", "nbody5 (config 1)"), ("nbody100", "nbody100 (config 2)"),
                          ("protein", "protein (config 3 shape)"), ("large", "large 1M (config 5, ONE GPU)")):
            try:
                table[tag] = quick_config(name, dev, flush)
            except Exception as exc:
                table[tag] = dict(error=f"{type(exc).__name__}: {exc}"[:300])
        line["per_config"] = table
    if not args.no_cpu_baseline and has_edges:
        torch.set_num_threads(cores)
        t_cpu = time_cpu(oracle_step_fn(data, hp, model=args.model), 1, 3)
        line["cpu_baseline"] = dict(value=E * LAYERS / t_cpu, unit="edges/s", cores=cores, kind="port",
                                    ms_per_step=t_cpu * 1e3,
                                    sample="the full workload: 1 warm-up + 3 timed training steps of oracle/ "
                                           "(CPU restatement of the reference's torch op chain)")
    if not args.no_gpu_eager_bar and has_edges:
        try:
            step = oracle_step_fn(data, hp, device=str(dev), model=args.model)

            def eager():
                step()
                torch.cuda.synchronize()
            t_eager = time_cpu(eager, 3, 10)
            line["gpu_eager_baseline"] = dict(value=E * LAYERS / t_eager, unit="edges/s", ms_per_step=t_eager * 1e3,
                                              kind="port", what="oracle/ (the reference's torch op chain: gather, cat, "
                                              "Linear, scatter_add, autograd, torch.optim.Adam) run eagerly in fp32 on "
                                              "this GPU, wall clock with a synchronize per step (BASELINE.md 3.5's GPU bar)")
        except Exception as exc:
            line["gpu_eager_baseline"] = dict(error=f"{type(exc).__name__}: {exc}"[:300])


def partition_setup(data, hp, args, world, rank, dev, device_graph):
    """This rank's share of ONE graph: (local host tensors, prebuilt slab graph or None, runner factory, MMD sample ids,
    MMD scales, transport name, owned edge count)."""
    from fastegnn_b200.partitioned import DeviceSlabPlan, PartitionedFastEGNN, SlabPlan
    N, C = int(data["loc_0"].size(0)), data["C"]
    gen = torch.Generator().manual_seed(0)
    ns = min(hp["sample"] * C, N)
    idx_glob = sample_indices([N], ns, gen)[0].tolist()
    if device_graph:
        plan = DeviceSlabPlan(data["loc_0"].to(dev), data["radius"], world, rank)   # every rank builds ITS slab's graph
        rows = plan.local_rows.cpu()
        local = {k: data[k][rows].contiguous() for k in ("node_feat", "loc_0", "vel_0", "loc_t")}
        graph, E_loc = plan.graph, plan.graph.E
        pos = torch.empty(N, dtype=torch.int64)
        pos[plan.order.cpu()] = torch.arange(N)
        mine = [int(plan.local_id[int(pos[g])]) for g in idx_glob if plan.owner[int(pos[g])] == rank]
    else:
        plan = SlabPlan(data["loc_0"].numpy(), data["edge_index"].numpy(), world)
        loc = plan.localize(rank, dict(node_feat=data["node_feat"].numpy(), loc_0=data["loc_0"].numpy(),
                                       vel_0=data["vel_0"].numpy(), loc_t=data["loc_t"].numpy()),
                            dict(edge_attr=data["edge_attr"].numpy()))
        local = {k: torch.from_numpy(v) for k, v in loc.items()}
        graph, E_loc = None, int(local["edge_index"].size(1))
        mine = [int(plan.local_id[g]) for g in idx_glob if plan.owner[g] == rank]
    local["loc_mean"] = data["loc_mean"]
    local.update(C=C, gravity=data["gravity"], sizes=[N], n_graphs=1)
    if graph is not None:
        local["edge_index"] = None
    idx_all = torch.tensor([mine], dtype=torch.int32).reshape(1, len(mine))
    scales = (1.0 if rank == 0 else 0.0, len(mine) / float(ns))
    used = dict(name=None)

    def factory(model):
        order = {"fused": ["fused", "p2p", "nccl"], "p2p": ["p2p", "nccl"], "nccl": ["nccl"]}[args.halo]
        last = None
        for h in order:                           # symmetric memory needs one NVLink domain; NCCL works everywhere
            try:
                r = PartitionedFastEGNN(model, plan, rank, dev, halo=h)
                used["name"] = h if h == args.halo else f"{h} (requested {args.halo}: {type(last).__name__})"
                return r
            except Exception as exc:              # noqa: BLE001 - the fallback is reported in the JSON line
                last = exc
        raise last
    names = {"fused": "fused payload+signal kernels over NVLink peer memory, deterministic reverse halo, one-shot all-reduce",
             "p2p": "peer-memory kernels over NVLink + symmetric-memory barrier", "nccl": "NCCL all-to-all"}
    return local, graph, factory, idx_all, scales, names[args.halo], E_loc


def partition_parity(world, rank, dev, halo, n=3000, C=8):
    """In-run parity of the partitioned path against ONE GPU on a small cloud (what tests/dist_check.py checks): worst
    relative error over the owned rows of x', Z', dL/dx0 and every weight gradient, max over ranks."""
    import torch.distributed as dist
    from fastegnn_b200 import CsrGraph, FastEGNN
    from fastegnn_b200.partitioned import DeviceSlabPlan, PartitionedFastEGNN
    data = make_cloud_device(n, 14.0, C, 5, None, None)
    g = torch.Generator().manual_seed(1)
    wx, wz = torch.randn(n, 3, generator=g).to(dev), torch.randn(1, 3, C, generator=g).to(dev)
    torch.manual_seed(3)
    model = FastEGNN(node_feat_nf=2, node_attr_nf=0, edge_attr_nf=2, hidden_nf=H, virtual_channels=C, device=dev, n_layers=3)
    with torch.no_grad():
        for k, p in model.named_parameters():     # natural magnitude on the coordinate path (default init: gain 1e-3)
            if k.endswith(".2.weight") and ("coord_mlp_r" in k or "coord_mlp_v_virtual" in k):
                p.mul_(300.0)
    t = {k: v.to(dev) for k, v in data.items() if torch.is_tensor(v)}
    x0 = t["loc_0"].clone().requires_grad_(True)
    gfull = CsrGraph.from_radius(t["loc_0"], t["batch"], 1, data["radius"], 0.0, 2)
    xr, Zr = model(node_feat=t["node_feat"], node_loc=x0, node_vel=t["vel_0"], edge_index=gfull, data_batch=t["batch"],
                   loc_mean=t["loc_mean"])
    ((xr * wx).sum() + (Zr * wz).sum()).backward()
    ref = {k: (None if p.grad is None else p.grad.clone()) for k, p in model.named_parameters()}
    ref_gx0 = x0.grad.clone()
    model.zero_grad(set_to_none=True)
    plan = DeviceSlabPlan(t["loc_0"], data["radius"], world, rank)
    rows = plan.local_rows
    runner = PartitionedFastEGNN(model, plan, rank, dev, halo=halo)
    Nn = runner.comm.N
    xl = t["loc_0"][rows].clone().requires_grad_(True)
    xo, Zo = runner(t["node_feat"][rows], xl, t["vel_0"][rows], plan.graph, t["loc_mean"], None, n_global=n)
    loss = (xo * wx[rows][:Nn]).sum() + ((Zo * wz).sum() if rank == 0 else 0.0 * Zo.sum())
    loss.backward()
    runner.allreduce_gradients()
    torch.cuda.synchronize()
    rel = lambda a, b: float((a.detach().double() - b.detach().double()).abs().max() / (b.detach().double().abs().max() + 1e-30))
    errs = [rel(xo, xr.detach()[rows[:Nn]]), rel(Zo, Zr.detach()), rel(xl.grad[:Nn], ref_gx0[rows[:Nn]])]
    errs += [rel(p.grad, ref[k]) for k, p in model.named_parameters() if ref[k] is not None]
    e = torch.tensor([max(errs)], device=dev, dtype=torch.float64)
    dist.all_reduce(e, op=dist.ReduceOp.MAX)
    return float(e[0])


def partitioned_block(args, world, rank, dev, flush, steps=5, warmup=3):
    """north_star item 5: ONE config-5 graph (1 M nodes, mean degree 30, C=8) in `world` slabs -- strong scaling against
    the same graph on one GPU, with the per-layer exchange times and an in-run parity figure."""
    import ctypes as Ct
    import torch.distributed as dist
    from fastegnn_b200 import CsrGraph, _lib as L
    n = args.part_nodes
    hp = dict(sigma=1.0, weight=0.01, sample=3)
    data = make_cloud_device(n, 30.0, 8, 0, None, None)
    t0 = time.perf_counter()
    local, graph, factory, idx_all, scales, halo_name, E_loc = partition_setup(data, hp, args, world, rank, dev, True)
    torch.cuda.synchronize()
    plan_s = time.perf_counter() - t0
    sb = StepBench(local, hp, dev, world=world, rank=rank, graph=graph, runner_factory=factory,
                   use_cuda_graph=not args.no_graph, n_global=n, idx_all=idx_all, mmd_scales=scales)
    comm = sb.runner.comm
    for _ in range(warmup):
        sb.resident()
    dist.barrier()
    torch.cuda.synchronize()
    ms = timed(sb.resident, steps, flush)
    tt = torch.tensor([ms], device=dev, dtype=torch.float64)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ee = torch.tensor([float(E_loc), float(comm.Nl - comm.N), float(E_loc), -float(E_loc)], device=dev, dtype=torch.float64)
    tot = ee.clone()
    dist.all_reduce(tot[:2])
    mx = ee[2:].clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    ms_n, E_all, halo_rows = float(tt[0]), float(tot[0]), float(tot[1])
    if hasattr(comm, "check"):
        comm.check()
    out = dict(workload=f"large: N={n} nodes, E={int(E_all)} directed edges, C=8, L={LAYERS}, ONE graph in {world} slabs; "
                        f"every rank builds its slab's radius graph on its device (plan + graph {plan_s:.2f} s, once), "
                        "CSR reused by every step in both arms",
               halo=halo_name, n_gpus=world, ms_per_step=ms_n, layer_edges_per_s=E_all * LAYERS / (ms_n * 1e-3),
               cuda_graph=sb.g is not None, steps=steps, warmup=warmup,
               edges_per_rank=dict(max=float(mx[0]), min=-float(mx[1]), mean=E_all / world),
               halo_rows_per_rank_mean=halo_rows / world,
               halo_bytes_per_layer_per_rank=int(comm.n_send * (4 * H + 12)))
    if sb.why:
        out["cuda_graph_error"] = sb.why
    # ---- the exchanges alone (CUDA events, max over ranks)
    try:
        from fastegnn_b200.partitioned import FusedHaloComm
        if isinstance(comm, FusedHaloComm):
            st = torch.cuda.current_stream().cuda_stream

            def push():
                L.check(L.lib.fegnn_halo_push_signal(Ct.byref(comm.p2p), 0, comm.n_send, L.ptr(comm.send_idx32), 0,
                                                     L.ptr(comm.fwd_q[0]), L.ptr(comm.fwd_x[0]), L.ptr(comm.Qs[0]),
                                                     L.ptr(comm.xs[0]), st), "halo_push_signal")
            buf = torch.zeros(3 * 8 + H * 8 + 3, device=dev)
            res = {}
            for name, fn in (("halo_push_signal_us", push), ("p2p_allreduce_us", lambda: comm.allreduce(buf))):
                for _ in range(5):
                    fn()
                dist.barrier()
                torch.cuda.synchronize()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                for _ in range(50):
                    fn()
                e.record()
                torch.cuda.synchronize()
                v = torch.tensor([s.elapsed_time(e) / 50 * 1e3], device=dev, dtype=torch.float64)
                dist.all_reduce(v, op=dist.ReduceOp.MAX)
                res[name] = round(float(v[0]), 2)
            res["per_step_us"] = round(2 * LAYERS * res["halo_push_signal_us"] + (2 * LAYERS + 2) * res["p2p_allreduce_us"], 1)
            res["limiting"] = "halo_push_signal (payload over NVLink + all-rank signal / wait)"
            res["what"] = ("one forward halo exchange of layer 0 (payload stores + signal + wait in ONE kernel) and one "
                           "one-shot all-reduce of 539 floats, 50 back-to-back calls each, max over ranks; a step has "
                           f"{2 * LAYERS} halo exchanges and {2 * LAYERS + 2} small all-reduces + one NCCL all-reduce of the "
                           "weight gradients")
            out["exchange"] = res
            comm.check()
    except Exception as exc:
        out["exchange"] = dict(error=f"{type(exc).__name__}: {exc}"[:300])
    del sb
    torch.cuda.empty_cache()
    # ---- the same graph on ONE GPU (rank 0; the others wait)
    ms1 = None
    if rank == 0:
        try:
            g1 = CsrGraph.from_radius(data["loc_0"].to(dev), data["batch"].to(dev), 1, data["radius"], 0.0, 2)
            sb1 = StepBench(data, hp, dev, graph=g1, use_cuda_graph=not args.no_graph)
            for _ in range(warmup):
                sb1.resident()
            ms1 = timed(sb1.resident, steps, flush)
            out["one_gpu"] = dict(ms_per_step=ms1, edges=int(g1.E), layer_edges_per_s=g1.E * LAYERS / (ms1 * 1e-3))
            out["strong_scaling_efficiency"] = ms1 / (world * ms_n)
            out["speedup"] = ms1 / ms_n
            del sb1, g1
        except Exception as exc:
            out["one_gpu"] = dict(error=f"{type(exc).__name__}: {exc}"[:300])
        torch.cuda.empty_cache()
    dist.barrier()
    torch.cuda.synchronize()
    # ---- in-run parity against one GPU (small cloud)
    try:
        halo = "fused" if halo_name.startswith("fused") else ("p2p" if halo_name.startswith("peer") else "nccl")
        out["parity_vs_one_gpu"] = dict(worst_rel_err=partition_parity(world, rank, dev, halo),
                                        what="3 000-node cloud, C=8, 3 layers: owned rows of x', Z', dL/dx0 and every "
                                             "weight gradient against the single-GPU path of the same module (default "
                                             "TF32 arithmetic in both), max over ranks")
    except Exception as exc:
        out["parity_vs_one_gpu"] = dict(error=f"{type(exc).__name__}: {exc}"[:300])
    return out


def rollout_profile(model, t, dev, E, flush, steps=20):
    """SURVEY.md 8 f4 (utils/train.py:24-27,191-192: evaluation epochs, backprop=False): the forward-only stack
    (fegnn_model_forward_inference: two ping-pong states + one shared block, nothing saved) as ONE CUDA graph, next to the
    training forward of the same batch (what model.eval() ran before the forward-only stack existed)."""
    kw = dict(node_feat=t["node_feat"], node_loc=t["loc_0"], node_vel=t["vel_0"], edge_index=t["edge_index"],
              data_batch=t["batch"], loc_mean=t["loc_mean"], edge_attr=t["edge_attr"])
    out = {}
    was_training = model.training
    try:
        order = (("forward_only", False), ("training_forward", True))
        if os.environ.get("FEGNN_ROLLOUT_ORDER") == "rev":
            order = order[::-1]
        for name, keep in order:
            model.eval()
            model.eval_keeps_graph = keep
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(3):
                    model(**kw)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats(dev)
            base = torch.cuda.memory_allocated(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                y = model(**kw)
            for _ in range(3):
                g.replay()
            ms = timed(g.replay, steps, flush)
            out[name] = dict(ms=round(ms, 4), layer_edges_per_s=E * LAYERS / (ms * 1e-3),
                             graph_pool_mb=round((torch.cuda.max_memory_allocated(dev) - base) / 2 ** 20, 1))
            del g, y
    finally:
        model.eval_keeps_graph = False
        model.train(was_training)
    out["what"] = "one captured 4-layer forward of the benchmark batch incl. graph prep, L2 flushed; graph_pool_mb = peak memory of the capture"
    return out


def graph_build_profile(data, t, dev, B, flush):
    """SURVEY.md 8 f2: the graph construction in front of the path (radius_graph + cutoff_edge + norm + the CSR sort) on
    the device, next to the CPU restatement (oracle/radius_graph_oracle.py: KD-tree candidates + numpy sorts)."""
    from fastegnn_b200 import CsrGraph
    from oracle import radius_graph_oracle as rgo
    r = data["radius"]
    out = {}
    for cr in (0.0, 0.5):
        for _ in range(3):
            g = CsrGraph.from_radius(t["loc_0"], t["batch"], B, r, cr, 2)
        ts = []
        for _ in range(10):
            flush.fill_(1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            g = CsrGraph.from_radius(t["loc_0"], t["batch"], B, r, cr, 2)       # includes its one host read of the count
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e))
        ms = sum(ts) / len(ts)
        cpu_ms, same = None, None
        if data["loc_0"].size(0) <= 200_000:                   # bounded CPU sample: the port takes minutes at 1e6 nodes
            t0 = time.perf_counter()
            o = rgo.radius_graph_csr(data["loc_0"].numpy(), np.concatenate([[0], np.cumsum(data["sizes"])]), r, cr)
            cpu_ms = round((time.perf_counter() - t0) * 1e3, 2)
            same = bool(o["row"].shape[0] == g.E and np.array_equal(g.col.cpu().numpy(), o["col"]))
        out[f"cutoff_rate={cr}"] = dict(edges=int(g.E), candidates=int(g.n_candidates), ms=round(ms, 4),
                                        edges_per_s=g.E / (ms * 1e-3), cpu_port_ms=cpu_ms, identical_to_oracle=same)
    out["what"] = ("CsrGraph.from_radius (fegnn_radius_graph_count + _fill, CUDA events incl. the host read of the "
                   "candidate count) vs oracle/radius_graph_oracle.py on 1 host thread")
    return out


def edge_bwd_at_scale(model, dev, flush, peak_tf, probes, peaks, name="water3d_b20"):
    """The same kernel on the reference's training batch (20 Water-3D graphs per step, main_simulation.py:46: 3.6e6 edges),
    where a launch is 190 tiles per SM instead of 9.6: the tile rate without the per-launch fixed costs."""
    import ctypes as Ct
    from fastegnn_b200 import _lib as L
    from fastegnn_b200.ops import CsrGraph, SavedBlock, layer_ptrs, make_dims
    data, _ = make_workload(name, 0, 0)
    t = {k: v.to(dev) for k, v in data.items() if torch.is_tensor(v)}
    N, E, B, C = t["loc_0"].size(0), t["edge_index"].size(1), data["n_graphs"], data["C"]
    graph = CsrGraph(t["edge_index"], t["batch"], t["edge_attr"], B)
    dims = make_dims(N, N, E, B, C, 2, L.F_GRAVITY if data["gravity"] is not None else 0, data["gravity"])
    named = dict(model.named_parameters())
    ptrs = layer_ptrs(named, "gcl_0")
    sv = SavedBlock(dims, dev)
    sv.view("P", (N, H)).normal_()
    sv.view("Q", (N, H)).normal_()
    gv = {k: torch.zeros_like(p) for k, p in named.items() if k.startswith("gcl_0.")}
    gr = layer_ptrs(gv, "gcl_0")
    gm, gt = torch.randn(N, H, device=dev), torch.randn(N, 3, device=dev)
    gP, gQ, gx = torch.empty(N, H, device=dev), torch.empty(N, H, device=dev), torch.zeros(N, 3, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    run = lambda: L.check(L.lib.fegnn_edge_backward(Ct.byref(dims), Ct.byref(graph.c), Ct.byref(ptrs), Ct.byref(gr), L.ptr(t["loc_0"]),
                                                    Ct.byref(sv.c), L.ptr(gm), L.ptr(gt), L.ptr(gP), L.ptr(gQ), L.ptr(gx), st))
    for _ in range(3):
        run()
    ts = []
    for _ in range(10):
        flush.fill_(1)
        s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s_.record(); run(); e_.record()
        torch.cuda.synchronize()
        ts.append(s_.elapsed_time(e_))
    t_s = sum(ts) / len(ts) * 1e-3
    flop = 6 * 2 * H * H * E
    out = dict(workload=f"{name}: N={N} nodes, E={E} edges (random P / Q / upstream gradients)", us=round(t_s * 1e6, 1),
               achieved=flop / t_s / 1e12, unit="TFLOP/s", frac=flop / t_s / 1e12 / peak_tf,
               edges_per_s=E / t_s)
    if "error" not in probes:
        algo_bytes = E * (4 + 4 + 4 * 2 + 2 * 256 + 24 + 12 + 256 + 2 * 268)
        t_model = max(flop / (probes["tcgen05_f16_tflops"] * 1e12), 3 * H * E / (probes["mufu_tanh_gops"] * 1e9),
                      algo_bytes / (peaks.get("hbm_gbs", 6650.0) * 1e9))
        out["frac_of_model"] = t_model / t_s
    try:                           # dram bytes of one ncu --set full capture of this launch (profiles/ncu_traffic_r2.json)
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic_r2.json")))
        out["traffic"] = tr.get(f"edge_bwd[mode=7]@E={E}")
    except Exception:
        out["traffic"] = None
    del sv, graph, t
    torch.cuda.empty_cache()
    return out


def phase_profile(model, t, dev, data, E, N, B, C, flush):
    """CUDA-event time of every phase of layer 0 (one C-ABI call each), and the roofline of the
    dominant kernel (edge backward)."""
    import ctypes as Ct
    from fastegnn_b200 import _lib as L
    from fastegnn_b200.layer_fn import LayerPhases
    from fastegnn_b200.ops import CsrGraph, layer_ptrs, make_dims
    lib = L.lib
    net = model
    st = torch.cuda.current_stream().cuda_stream
    graph = CsrGraph(t["edge_index"], t["batch"], t["edge_attr"], B)
    flags = L.F_GRAVITY if data["gravity"] is not None else 0
    dims = make_dims(N, N, E, B, C, 2, flags, data["gravity"])
    named = dict(model.named_parameters())
    ptrs = layer_ptrs(named, "gcl_0")
    ph = LayerPhases(dims, graph, ptrs, dev)
    h = torch.nn.functional.linear(t["node_feat"], model.embedding_in.weight, model.embedding_in.bias).detach()
    x, v, Z = t["loc_0"], t["vel_0"], t["loc_mean"]
    S = model.virtual_node_feat.detach()[0].T.contiguous().unsqueeze(0).repeat(B, 1, 1).contiguous()
    xsum = torch.zeros(B, 3, device=dev).index_add_(0, t["batch"], x)
    e32 = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float32)
    gviews = {k: torch.zeros_like(p) for k, p in named.items() if k.startswith("gcl_0.")}
    gr = layer_ptrs(gviews, "gcl_0")
    pd, pg, pp, ps, pgr = Ct.byref(dims), Ct.byref(graph.c), Ct.byref(ptrs), Ct.byref(ph.saved.c), Ct.byref(gr)
    x_new, xsum_new, h_new, Z_new, S_new = e32(N, 3), e32(B, 3), e32(N, H), e32(B, 3, C), e32(B, C, H)
    gZ, gS, gDsum, gUsum = e32(B, 3, C), e32(B, C, H), e32(B, 3, C), e32(B, C, H)
    gh, gzh1, gm, gu = torch.randn(N, H, device=dev), e32(N, H), e32(N, H), e32(N, C, H)
    gxn, gAv, gG1, gx, gsv, gsg, gt = torch.randn(N, 3, device=dev), e32(N, H), e32(B, C, H), e32(N, 3), e32(N), e32(N), e32(N, 3)
    gP, gQ, gxs = e32(N, H), e32(N, H), e32(B, 3)
    gZn, gSn = torch.randn(B, 3, C, device=dev), torch.randn(B, C, H, device=dev)
    p = L.ptr
    calls = [
        ("graph_prep", lambda: CsrGraph(t["edge_index"], t["batch"], t["edge_attr"], B)),
        ("graph_pre_fwd", lambda: lib.fegnn_graph_pre_forward(pd, pg, pp, p(Z), p(S), p(xsum), ps, st)),
        ("node_pre_fwd", lambda: lib.fegnn_node_pre_forward(pd, pp, p(h), ps, st)),
        ("edge_fwd", lambda: lib.fegnn_edge_forward(pd, pg, pp, p(x), ps, st)),
        ("virtual_fwd", lambda: lib.fegnn_virtual_forward(pd, pg, pp, p(x), p(v), p(Z), ps, p(x_new), p(xsum_new), st)),
        ("node_h_fwd", lambda: lib.fegnn_node_h_forward(pd, pg, pp, p(h), ps, p(h_new), st)),
        ("graph_post_fwd", lambda: lib.fegnn_graph_post_forward(pd, pg, pp, p(Z), p(S), ps, p(Z_new), p(S_new), st)),
        ("graph_post_bwd", lambda: lib.fegnn_graph_post_backward(pd, pg, pp, pgr, p(S), ps, p(gZn), p(gSn), p(gZ), p(gS),
                                                                 p(gDsum), p(gUsum), st)),
        ("node_h_bwd", lambda: lib.fegnn_node_h_backward(pd, pg, pp, pgr, ps, p(gh), p(gzh1), p(gm), p(gu), st)),
        ("virtual_bwd", lambda: lib.fegnn_virtual_backward(pd, pg, pp, pgr, p(x), p(v), p(Z), ps, p(gxn), None, p(gDsum),
                                                           p(gUsum), p(gu), p(gAv), p(gG1), p(gx), p(gZ), p(gsv), p(gsg),
                                                           p(gt), st)),
        ("edge_bwd", lambda: lib.fegnn_edge_backward(pd, pg, pp, pgr, p(x), ps, p(gm), p(gt), p(gP), p(gQ), p(gx), st)),
        ("graph_pre_bwd", lambda: lib.fegnn_graph_pre_backward(pd, pg, pp, pgr, p(S), ps, p(gG1), p(gS), p(gZ), p(gxs), st)),
        ("node_pre_bwd", lambda: lib.fegnn_node_pre_backward(pd, pp, pgr, p(h), p(gP), p(gQ), p(gAv), p(gzh1), p(gsv),
                                                             p(gsg), p(gh), st)),
    ]
    out = {}

    def with_mode(phase, mode, fn):
        def run():
            old = L.get_mode(phase)
            L.set_mode(phase, mode)
            try:
                return fn()
            finally:
                L.set_mode(phase, old)
        return run
    edge_fwd_fn = dict(calls)["edge_fwd"]
    calls += [(f"edge_fwd[mode={m}]", with_mode("edge_forward", m, edge_fwd_fn)) for m in (0, 1, 3)]
    virt_fwd_fn, virt_bwd_fn = dict(calls)["virtual_fwd"], dict(calls)["virtual_bwd"]
    calls += [(f"virtual_fwd[mode={m}]", with_mode("virtual_forward", m, virt_fwd_fn)) for m in (0, 1)]
    calls += [(f"virtual_bwd[mode={m}]", with_mode("virtual_backward", m, virt_bwd_fn)) for m in (0, 1)]
    npre_fn = dict(calls)["node_pre_fwd"]
    calls += [(f"node_pre_fwd[mode={m}]", with_mode("node_forward", m, npre_fn)) for m in (0, 1)]
    if "node_h_fwd" in dict(calls):
        nh_fn = dict(calls)["node_h_fwd"]
        calls += [(f"node_h_fwd[mode={m}]", with_mode("node_forward", m, nh_fn)) for m in (0, 3)]
    edge_bwd_fn = dict(calls)["edge_bwd"]
    calls += [(f"edge_bwd[mode={m}]", with_mode("edge_backward", m, edge_bwd_fn)) for m in (0, 1, 2, 4, 5, 7, 8)]
    for name, fn in calls:
        for _ in range(3):
            fn()
        ts = []
        for _ in range(10):
            flush.fill_(1)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); fn(); e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e))
        out[name] = round(sum(ts) / len(ts), 4)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops", 1590.0)
    which = "measured (MEASURED_PEAKS.json bf16_tflops, burst: kernel timed alone)" if "bf16_tflops" in peaks else "fallback 1590"
    # ---- the pipes this formulation runs on, measured live on this GPU (fegnn_peak_probe, csrc/peak_probe.cu)
    probes = {}
    try:
        sink = torch.zeros(4, device=dev)
        for kind, key, iters, unit in ((0, "tcgen05_tf32_tflops", 16384, 1e12), (1, "tcgen05_f16_tflops", 16384, 1e12),
                                       (2, "ffma_fp32_tflops", 8192, 1e12), (3, "mufu_tanh_gops", 4096, 1e9)):
            ops = Ct.c_double(0.0)
            run = lambda: L.check(lib.fegnn_peak_probe(kind, iters, p(sink), Ct.byref(ops), st), "fegnn_peak_probe")
            for _ in range(2):
                run()
            best = 1e30
            for _ in range(5):
                s_, e_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s_.record(); run(); e_.record()
                torch.cuda.synchronize()
                best = min(best, s_.elapsed_time(e_))
            probes[key] = round(ops.value / (best * 1e-3) / unit, 1)
        probes["what"] = ("one launch each, best of 5 (burst): tcgen05.mma cta_group::1 M128 N256 from shared-memory operands "
                          "(kind::tf32 K8 / kind::f16 K16) issued by one thread per SM on 148 SMs -- the instruction form "
                          "of the edge / virtual kernels; FFMA and MUFU tanh.approx with 8 independent chains per thread")
    except Exception as exc:
        probes = dict(error=f"{type(exc).__name__}: {exc}"[:300])
    bwd_mode = L.get_mode("edge_backward")
    if bwd_mode == 6:              # auto (fegnn.h): the packed-fp16 two-stream kernel wherever the tensor-core form applies
        bwd_mode = 7
    flop = 6 * 2 * H * H * E       # recompute 2 + dgrad 2 + wgrad 2 GEMMs of [E,64]x[64,64]; bias-sum GEMM columns not counted
    t_s = out["edge_bwd"] * 1e-3
    ach = flop / t_s / 1e12
    traffic = None
    try:                           # dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture, per launch
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic_r2.json")))
        traffic = tr.get(f"edge_bwd[mode={bwd_mode}]@E={E}")
    except Exception:
        pass
    algo_bytes = E * (4 + 4 + 4 * 2 + 2 * 256 + 24 + 12 + 256 + 2 * 268)    # no-reuse model, SURVEY.md 8(d): ~1.35 KB/edge
    kname = {7: "bwd4::edge_bwd_tc4_kernel<2> (tcgen05 kind::f16 operands, packed-fp16 epilogues, two 128-edge tiles in flight per SM)",
             8: "bwd4::edge_bwd_tc4_kernel<4> (as <2> with 512 threads per tile)",
             5: "bwd3::edge_bwd_tc3_kernel (tcgen05 kind::f16, two 128-edge tiles in flight per SM)",
             4: "bwd2::edge_bwd_tc2_kernel<4> (tcgen05 TF32)", 2: "bwd2::edge_bwd_tc2_kernel<2> (tcgen05 TF32)",
             1: "edge_bwd_tc_kernel (tcgen05 TF32)", 0: "edge_bwd_kernel (fp32 FMA)"}[bwd_mode]
    model = None
    if "error" not in probes:
        pk = probes["tcgen05_f16_tflops"] if bwd_mode in (5, 7, 8) else (probes["tcgen05_tf32_tflops"] if bwd_mode else probes["ffma_fp32_tflops"])
        t_tensor = flop / (pk * 1e12)
        t_mufu = 3 * H * E / (probes["mufu_tanh_gops"] * 1e9)            # one tanh.approx per SiLU': z1, z2, z3 of every edge
        t_mem = algo_bytes / (peaks.get("hbm_gbs", 6650.0) * 1e9)
        t_model = max(t_tensor, t_mufu, t_mem)
        model = dict(t_tensor_us=round(t_tensor * 1e6, 2), t_mufu_us=round(t_mufu * 1e6, 2), t_mem_us=round(t_mem * 1e6, 2),
                     t_measured_us=round(t_s * 1e6, 2), frac_of_model=t_model / t_s,
                     what="SURVEY.md 8(d): max(t_tensor, t_mufu, t_mem) / t_measured with the tensor and MUFU rates "
                          "measured by the probes above and the no-reuse byte model against the measured HBM copy rate")
    at_scale = None
    try:
        at_scale = edge_bwd_at_scale(net, dev, flush, peak_tf, probes, peaks)
    except Exception as exc:
        at_scale = dict(error=f"{type(exc).__name__}: {exc}"[:300])
    roof = dict(kernel=f"{kname}, one launch = all E edges of one layer; CUDA events around the C-ABI call incl. its two "
                       "output memsets, L2 flushed",
                bound="tensor", achieved=ach, peak=peak_tf, unit="TFLOP/s", frac=ach / peak_tf, traffic=traffic,
                peak_source=which, peaks_measured=probes,
                peak_tf32_measured=probes.get("tcgen05_tf32_tflops"), peak_f16_measured=probes.get("tcgen05_f16_tflops"),
                peak_mufu_measured=probes.get("mufu_tanh_gops"), model=model, at_scale=at_scale,
                note="algorithmic flops = 6 GEMMs x 2*64*64 = 49152 per edge (the per-edge MLP recompute, its data gradient "
                     f"and its weight gradient); the no-reuse byte model is {algo_bytes / 1e6:.0f} MB per launch = "
                     f"{algo_bytes / t_s / 1e9:.0f} GB/s at this duration, under the HBM roof, and P/Q/x rows are L2-resident "
                     "at this size; `peak` is the cuBLAS bf16 figure of MEASURED_PEAKS.json (the cross-kernel denominator), "
                     "`peaks_measured` are the rates of the instruction forms this kernel actually issues")
    return dict(roofline=roof, phases_ms_layer0=out)


if __name__ == "__main__":
    main()
