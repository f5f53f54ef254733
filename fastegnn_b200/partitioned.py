"""Spatially partitioned FastEGNN for ONE large graph across the GPUs of a box (SURVEY.md 5.1 mode 2).

The reference has no distributed code; this is the multi-GPU form of the same layer
(models/FastEGNN.py:192-223).  Nodes are split into 1-D slabs along the longest axis (equal node
counts); a node is owned by one rank, an edge (row=i, col=j) by the owner of i -- the end every
reference aggregation reduces over (:127-129,:156).  Per layer:

  forward   node_pre -> HALO EXCHANGE of (Q_j, x_j) for remote cols j -> edge phase -> virtual phase
            -> ALL-REDUCE of the per-graph partial sums (Dsum 3C, Usum CH, xsum 3 floats per graph)
            -> node_h, graph_post (replicated)
  backward  graph_post_bwd (replicated) -> node_h_bwd -> virtual_bwd -> edge_bwd
            -> REVERSE HALO (remote dQ_j, dx_j summed at the owner) + ALL-REDUCE of (dG1, dZ) partials
            -> graph_pre_bwd (replicated) -> node_pre_bwd
  per step  one all-reduce of the flat weight-gradient buffer.

Collectives go through torch.distributed (NCCL over NVLink on the box, gloo in the CPU tests of the
host logic); all arithmetic is the same C-ABI phase calls as on one GPU (layer_fn.LayerPhases).
The total loss is the SUM over ranks of rank-local losses: terms that depend only on the replicated
virtual coordinates Z must be added on one rank (or divided by the world size).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _lib as L
from .layer_fn import LayerPhases
from .ops import CsrGraph, _on, _require_cuda, _stream, layer_ptrs, make_dims

lib = L.lib


# ------------------------------------------------------------------------------------- host-side plan
class SlabPlan:
    """Index bookkeeping of the slab partition (numpy, host).  Pure integer logic -- unit-tested on CPU."""

    def __init__(self, x: np.ndarray, edge_index: np.ndarray, world: int):
        x = np.asarray(x)
        ei = np.asarray(edge_index)
        N = x.shape[0]
        self.world, self.N = world, N
        self.axis = int(np.argmax(x.max(0) - x.min(0)))
        self.order = np.argsort(x[:, self.axis], kind="stable")            # global ids in slab order
        self.bounds = np.array([N * k // world for k in range(world + 1)], dtype=np.int64)
        self.owner = np.empty(N, dtype=np.int32)
        self.local_id = np.empty(N, dtype=np.int64)
        for k in range(world):
            ids = self.order[self.bounds[k]:self.bounds[k + 1]]
            self.owner[ids] = k
            self.local_id[ids] = np.arange(ids.size)
        row, col = ei[0], ei[1]
        self.edge_owner = self.owner[row]
        self.parts: List[Dict[str, np.ndarray]] = []
        halos = []
        for k in range(world):
            eidx = np.nonzero(self.edge_owner == k)[0]                      # keeps the caller's edge order
            r, c = row[eidx], col[eidx]
            remote = self.owner[c] != k
            hg = np.unique(c[remote])                                       # halo nodes (global ids) ...
            key = self.owner[hg].astype(np.int64) * N + self.local_id[hg]   # ... ordered by (owner rank, owner-local id)
            hg = hg[np.argsort(key, kind="stable")]
            halos.append(hg)
            n_own = int(self.bounds[k + 1] - self.bounds[k])
            halo_pos = {int(g): n_own + j for j, g in enumerate(hg)} if hg.size < 4096 else None
            col_local = self.local_id[c].copy()
            if hg.size:
                lut = np.full(N, -1, dtype=np.int64)
                lut[hg] = n_own + np.arange(hg.size)
                col_local[remote] = lut[c[remote]]
            self.parts.append(dict(edge_ids=eidx, row=self.local_id[r], col=col_local, n_own=n_own,
                                   owned=self.order[self.bounds[k]:self.bounds[k + 1]], halo=hg,
                                   recv_counts=np.bincount(self.owner[hg], minlength=world).astype(np.int64)))
        # what every rank must SEND: for destination d, the nodes of d's halo that this rank owns, in d's halo order
        for k in range(world):
            send_idx, send_counts = [], []
            for d in range(world):
                hg = halos[d]
                mine = hg[self.owner[hg] == k] if hg.size else hg
                send_idx.append(self.local_id[mine])
                send_counts.append(mine.size)
            self.parts[k]["send_idx"] = np.concatenate(send_idx).astype(np.int64) if send_idx else np.zeros(0, np.int64)
            self.parts[k]["send_counts"] = np.array(send_counts, dtype=np.int64)

    def localize(self, rank: int, node_arrays: Dict[str, np.ndarray], edge_arrays: Dict[str, np.ndarray]):
        """Slice global per-node / per-edge arrays for `rank`.  Node arrays get owned rows followed by halo rows."""
        p = self.parts[rank]
        ids = np.concatenate([p["owned"], p["halo"]])
        out = {k: np.ascontiguousarray(np.asarray(v)[ids]) for k, v in node_arrays.items()}
        out.update({k: np.ascontiguousarray(np.asarray(v)[p["edge_ids"]]) for k, v in edge_arrays.items()})
        out["edge_index"] = np.stack([p["row"], p["col"]]).astype(np.int64)
        return out


class DeviceSlabPlan:
    """The slab partition of a point cloud + radius graph, built by EVERY RANK FOR ITS OWN SLAB on its own device
    (SURVEY.md 8(e) / 8 f2) -- no rank ever holds the global edge list (3e7 edges at config 5).

    All ranks hold the cloud x [N,3] (12 MB at 1e6 nodes).  It is sorted along its longest axis (stable), rank k owns the
    sorted positions [N k / world, N (k+1) / world).  Rank k gathers its owned points plus every point whose axis
    coordinate lies within r of its slab (the only possible remote neighbours -- two contiguous runs of the sorted
    order), builds THAT sub-cloud's radius graph with fegnn_radius_graph_* (CsrGraph.from_radius; the CSR rows of the owned
    points are its prefix), keeps the candidates that are actually referenced as its halo (ascending sorted position ==
    ascending (owner rank, owner-local id)), and renumbers cols to [owned | halo].  The halo lists (a few 10^4 ids per
    rank) are all-gathered so that every rank can derive what it must send and every peer-memory address table.
    Node ids inside the plan are SORTED POSITIONS; `order` maps them to the caller's node ids.

    Exposes the same fields as SlabPlan (`world`, `N`, `owner`, `local_id`, `parts[k]` with n_own / halo / recv_counts and,
    for this rank, send_idx / send_counts), so HaloComm and the address-table builders work with either."""

    def __init__(self, x: torch.Tensor, r: float, world: int, rank: int, group=None, edge_attr_nf: int = 2,
                 build_graph=None):
        dev = x.device
        N = int(x.size(0))
        self.world, self.rank, self.N, self.r = world, rank, N, float(r)
        ext = x.max(0).values - x.min(0).values
        self.axis = int(torch.argmax(ext))
        key_all = x[:, self.axis].contiguous()
        self.order = torch.argsort(key_all, stable=True)                    # sorted position -> caller's node id
        xs = x[self.order].contiguous()
        key = xs[:, self.axis].contiguous()
        b = [N * k // world for k in range(world + 1)]
        self.bounds = np.array(b, dtype=np.int64)
        b0, b1 = b[rank], b[rank + 1]
        n_own = b1 - b0
        if n_own > 0:
            pad = float(r) * (1.0 + 1e-5) + 1e-30                           # candidates may be a superset (strict d2 < r2 test later)
            lo, hi = key[b0] - pad, key[b1 - 1] + pad
            s_lo = int(torch.searchsorted(key, lo.reshape(1), right=False))
            s_hi = int(torch.searchsorted(key, hi.reshape(1), right=True))
            s_lo, s_hi = min(s_lo, b0), max(s_hi, b1)
        else:
            s_lo, s_hi = b0, b1
        cand_gid = torch.cat([torch.arange(s_lo, b0, device=dev), torch.arange(b1, s_hi, device=dev)])
        cloud = torch.cat([xs[b0:b1], xs[s_lo:b0], xs[b1:s_hi]]).contiguous()
        if build_graph is None:
            g = CsrGraph.from_radius(cloud, torch.zeros(cloud.size(0), dtype=torch.int64, device=dev), 1, r, 0.0,
                                     edge_attr_nf)
        else:
            g = build_graph(cloud)                                           # CPU tests inject the numpy oracle here
        E_own = int(g.rowptr[n_own]) if n_own > 0 else 0
        col = g.col[:E_own].long()
        used = torch.zeros(cand_gid.numel() + 1, dtype=torch.bool, device=dev)
        remote = col >= n_own
        used[(col[remote] - n_own)] = True
        used = used[:cand_gid.numel()]
        newid = torch.cumsum(used.to(torch.int64), 0) - 1 + n_own
        if cand_gid.numel():
            col = torch.where(remote, newid[(col - n_own).clamp(min=0)], col)
        halo_gid = cand_gid[used]
        n_halo = int(halo_gid.numel())
        # ---- this rank's graph in kernel layout: rows = owned, cols = [owned | halo]
        g.N, g.Nl, g.E = n_own, n_own + n_halo, E_own
        g.row, g.col = g.row[:E_own].contiguous(), col.to(torch.int32).contiguous()
        g.edge_attr = g.edge_attr[:E_own].contiguous() if g.Fe else g.edge_attr
        g.batch, g.dinv, g.rowptr = g.batch[:n_own].contiguous(), g.dinv[:n_own].contiguous(), g.rowptr[:n_own + 1].contiguous()
        g.inv_nb = torch.full((1,), 1.0 / max(1, N), device=dev, dtype=torch.float32)    # graph size is global
        if hasattr(g, "rebind"):
            g.rebind()
        self.graph = g
        self.local_rows = self.order[torch.cat([torch.arange(b0, b1, device=dev), halo_gid])]   # caller's ids: owned | halo
        # ---- halo lists of every rank (small): all-gather, padded to the longest
        if world > 1:
            cnt = torch.tensor([n_halo], dtype=torch.int64, device=dev)
            cnts = [torch.zeros_like(cnt) for _ in range(world)]
            dist.all_gather(cnts, cnt, group=group)
            cnts = [int(c) for c in cnts]
            m = max(max(cnts), 1)
            mine = torch.full((m,), -1, dtype=torch.int64, device=dev)
            mine[:n_halo] = halo_gid
            allh = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(allh, mine, group=group)
            halos = [h[:c].cpu().numpy() for h, c in zip(allh, cnts)]
        else:
            halos = [halo_gid.cpu().numpy()]
        ids = np.arange(N, dtype=np.int64)
        self.owner = (np.searchsorted(self.bounds, ids, side="right") - 1).astype(np.int32)
        self.local_id = ids - self.bounds[self.owner]
        self.parts: List[Dict[str, np.ndarray]] = []
        for k in range(world):
            hg = halos[k]
            self.parts.append(dict(n_own=int(b[k + 1] - b[k]), halo=hg,
                                   recv_counts=np.bincount(self.owner[hg], minlength=world).astype(np.int64)))
        send_idx, send_counts = [], []
        for d in range(world):
            hg = halos[d]
            mine_ = hg[self.owner[hg] == rank] if hg.size else hg
            send_idx.append(self.local_id[mine_])
            send_counts.append(mine_.size)
        self.parts[rank]["send_idx"] = np.concatenate(send_idx).astype(np.int64)
        self.parts[rank]["send_counts"] = np.array(send_counts, dtype=np.int64)
        for k in range(world):                                               # every rank's send_counts follow from recv_counts
            if k != rank:
                self.parts[k]["send_counts"] = np.array([int(self.parts[d]["recv_counts"][k]) for d in range(world)],
                                                        dtype=np.int64)


class HaloComm:
    """Device-side halo exchange + small all-reduces for one rank (hooks of LayerPhases)."""

    def __init__(self, plan: SlabPlan, rank: int, device, group=None):
        p = plan.parts[rank]
        self.N, self.Nl = p["n_own"], p["n_own"] + int(p["halo"].size)
        self.send_idx = torch.from_numpy(p["send_idx"]).to(device)
        self.send_counts = [int(v) for v in p["send_counts"]]
        self.recv_counts = [int(v) for v in p["recv_counts"]]
        self.n_send, self.n_recv = int(sum(self.send_counts)), int(sum(self.recv_counts))
        self.group, self.device = group, device
        self.world = plan.world

    # -- forward: owner -> users
    def exchange(self, Q: torch.Tensor, x: torch.Tensor) -> None:
        """Fill rows [N, Nl) of Q [Nl,64] and x [Nl,3] with the owners' current rows (one all-to-all)."""
        send = torch.cat([Q.index_select(0, self.send_idx), x.index_select(0, self.send_idx)], dim=1)
        recv = torch.empty(self.n_recv, send.size(1), device=self.device, dtype=torch.float32)
        dist.all_to_all_single(recv, send, self.recv_counts, self.send_counts, group=self.group)
        if self.n_recv:
            Q[self.N:] = recv[:, :L.H]
            x[self.N:] = recv[:, L.H:]

    # -- backward: users -> owner, summed
    def reduce_back(self, gQ: torch.Tensor, gx: torch.Tensor) -> None:
        send = torch.cat([gQ[self.N:], gx[self.N:]], dim=1).contiguous()
        recv = torch.empty(self.n_send, send.size(1), device=self.device, dtype=torch.float32)
        dist.all_to_all_single(recv, send, self.send_counts, self.recv_counts, group=self.group)
        if self.n_send:
            gQ.index_add_(0, self.send_idx, recv[:, :L.H])
            gx.index_add_(0, self.send_idx, recv[:, L.H:])

    def allreduce(self, *tensors: torch.Tensor) -> None:
        """Sum small per-graph tensors over ranks in ONE collective (rank order is fixed by the backend)."""
        flat = torch.cat([t.reshape(-1) for t in tensors])
        dist.all_reduce(flat, group=self.group)
        o = 0
        for t in tensors:
            n = t.numel()
            t.copy_(flat[o:o + n].view_as(t))
            o += n

    # LayerPhases hooks ---------------------------------------------------------------------------
    def after_node_pre(self, ph: LayerPhases, x: torch.Tensor) -> None:
        self.exchange(ph.saved.view("Q", (self.Nl, L.H)), x)

    def after_virtual(self, ph: LayerPhases, xsum_new: torch.Tensor) -> None:
        d = ph.d
        self.allreduce(ph.saved.view("Dsum", (d.B, 3, d.C)), ph.saved.view("Usum", (d.B, d.C, L.H)), xsum_new)

    def after_edge_backward(self, ph: LayerPhases, gQ, gx, gG1, gZ_part) -> None:
        self.reduce_back(gQ, gx)
        self.allreduce(gG1, gZ_part)


def p2p_address_tables(plan: SlabPlan, rank: int, n_layers: int, nl_max: int, base_q, base_x, base_gq, base_gx,
                       row_bytes_q: int = 4 * L.H, row_bytes_x: int = 12):
    """Destination byte addresses of the peer-memory halo kernels for `rank` (pure integer logic, unit-tested on the CPU
    against a simulated address space).  base_* [world] = every rank's base address of its symmetric Q [L, nl_max, 64],
    x [L, nl_max, 3], gQ [nl_max, 64] and gx [2, nl_max, 3] arrays.  Returns int64 numpy arrays
        fwd_q, fwd_x [L][n_send]   where send entry k (grouped by destination, in the destination's halo order) lands,
        bwd_q [n_recv], bwd_x [2][n_recv]   the owner's row of each of this rank's halo rows (gx has two slots)."""
    parts = plan.parts
    dst_row, dst_rank = [], []
    for d in range(plan.world):
        cnt = int(parts[rank]["send_counts"][d])
        off = int(parts[d]["recv_counts"][:rank].sum())                # d's halo is ordered by (owner rank, owner-local id)
        dst_row.append(parts[d]["n_own"] + off + np.arange(cnt, dtype=np.int64))
        dst_rank.append(np.full(cnt, d, dtype=np.int64))
    dst_row = np.concatenate(dst_row) if dst_row else np.zeros(0, np.int64)
    dst_rank = np.concatenate(dst_rank) if dst_rank else np.zeros(0, np.int64)
    bq, bx = np.asarray(base_q, dtype=np.int64)[dst_rank], np.asarray(base_x, dtype=np.int64)[dst_rank]
    fwd_q = [bq + (l * nl_max + dst_row) * row_bytes_q for l in range(n_layers)]
    fwd_x = [bx + (l * nl_max + dst_row) * row_bytes_x for l in range(n_layers)]
    hg = parts[rank]["halo"]
    own, lid = plan.owner[hg].astype(np.int64), plan.local_id[hg].astype(np.int64)
    bwd_q = np.asarray(base_gq, dtype=np.int64)[own] + lid * row_bytes_q
    bgx = np.asarray(base_gx, dtype=np.int64)[own]
    bwd_x = [bgx + (slot * nl_max + lid) * row_bytes_x for slot in range(2)]
    return fwd_q, fwd_x, bwd_q, bwd_x


class P2PHaloComm(HaloComm):
    """Halo exchange by direct peer-memory access over NVLink / NVSwitch (csrc/halo.cu) instead of NCCL all-to-all.

    Q and x of every layer, and the gradient buffers gQ / gx, live in torch symmetric memory, so every rank can address
    its peers' arrays.  Forward: ONE kernel stores the owners' (Q_j, x_j) rows straight into the users' halo rows, then a
    symmetric-memory barrier on the stream.  Backward: barrier, ONE kernel adds the users' (dQ_j, dx_j) halo rows into the
    owners' rows with remote atomics, barrier.  Destination addresses are fixed by the plan and precomputed as 64-bit
    tables.  The tiny per-graph all-reduces stay on NCCL.  Measured on 2 B200 (tools/p2p_probe.py, 6 000 rows): 20 us per
    exchange against 90 us for index_select + cat + all_to_all_single + two slice copies."""

    def __init__(self, plan: SlabPlan, rank: int, device, n_layers: int, group=None):
        super().__init__(plan, rank, device, group)
        import torch.distributed._symmetric_memory as symm
        grp = dist.group.WORLD if group is None else group
        parts = plan.parts
        self.n_layers = n_layers
        self.Nl_max = Nm = max(int(p["n_own"] + p["halo"].size) for p in parts)
        f32 = dict(dtype=torch.float32, device=device)
        self.Qs, self.xs = symm.empty(n_layers, Nm, L.H, **f32), symm.empty(n_layers, Nm, 3, **f32)
        self.gQs, self.gxs = symm.empty(Nm, L.H, **f32), symm.empty(2, Nm, 3, **f32)
        self.hQ, self.hx = symm.rendezvous(self.Qs, grp), symm.rendezvous(self.xs, grp)
        self.hgQ, self.hgx = symm.rendezvous(self.gQs, grp), symm.rendezvous(self.gxs, grp)
        for t in (self.Qs, self.xs, self.gQs, self.gxs):
            t.zero_()
        i64 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(device)
        fq, fx, bq, bx = p2p_address_tables(plan, rank, n_layers, Nm, self.hQ.buffer_ptrs, self.hx.buffer_ptrs,
                                            self.hgQ.buffer_ptrs, self.hgx.buffer_ptrs)
        self.send_idx32 = self.send_idx.to(torch.int32)
        self.fwd_q, self.fwd_x = [i64(a) for a in fq], [i64(a) for a in fx]
        self.bwd_q, self.bwd_x = i64(bq), [i64(a) for a in bx]
        self._slot = 0
        self._layer_of = {}

    def barrier(self) -> None:
        self.hQ.barrier(channel=0)

    # -- forward
    def bind_layer(self, ph: LayerPhases, layer: int) -> None:
        """This layer's Q is the symmetric array (node_pre writes the owned rows there, peers write the halo rows)."""
        ph.saved.c.Q = self.Qs[layer].data_ptr()
        self._layer_of[id(ph)] = layer

    def layer_x(self, layer: int, x: torch.Tensor, rows: int) -> torch.Tensor:
        """The layer's input coordinates inside symmetric memory ([Nl,3] view); `rows` leading rows of x are copied."""
        xs = self.xs[layer, :self.Nl]
        xs[:rows].copy_(x[:rows])
        return xs

    def after_node_pre(self, ph: LayerPhases, x: torch.Tensor) -> None:
        l = self._layer_of[id(ph)]
        L.check(lib.fegnn_halo_push(self.n_send, L.ptr(self.send_idx32), L.ptr(self.fwd_q[l]), L.ptr(self.fwd_x[l]),
                                    L.ptr(self.Qs[l]), L.ptr(x), _stream()), "fegnn_halo_push")
        self.barrier()

    # -- backward
    def grad_halo_buffers(self, ph: LayerPhases):
        self._slot ^= 1
        return self.gQs[:self.Nl], self.gxs[self._slot, :self.Nl]

    def after_edge_backward(self, ph: LayerPhases, gQ, gx, gG1, gZ_part) -> None:
        self.barrier()                       # every rank has zero-filled and accumulated its own gQ / gx of this layer
        L.check(lib.fegnn_halo_reduce_push(self.n_recv, self.N, L.ptr(self.bwd_q), L.ptr(self.bwd_x[self._slot]),
                                           L.ptr(gQ), L.ptr(gx), _stream()), "fegnn_halo_reduce_push")
        self.barrier()
        self.allreduce(gG1, gZ_part)


def fused_halo_tables(plan, rank: int, n_layers: int, nl_max: int, recv_cap: int, base_q, base_x, base_rq, base_rx,
                      row_bytes_q: int = 4 * L.H, row_bytes_x: int = 12):
    """Address / index tables of the fused (payload + signal) halo kernels for `rank` -- pure integer logic, unit-tested on
    the CPU against a simulated address space.  base_q / base_x [world]: every rank's symmetric Q [L, nl_max, 64] and
    x [L, nl_max, 3]; base_rq / base_rx [world]: every rank's RECEIVE buffers [2, recv_cap, 64] / [2, recv_cap, 3] of the
    reverse halo, whose slot k belongs to the owner's send entry k (entries grouped by user rank, in the user's halo order).
    Returns
        fwd_q, fwd_x [L][n_send]      where send entry k lands (the forward tables of p2p_address_tables),
        bwd_q, bwd_x [2][n_recv]      the slot, in the owner's receive buffer of either parity, of each halo row of `rank`,
        rows [n_b], ptr [n_b + 1], slots [n_send]   per owned boundary row: its receive slots in (user rank, halo order)
                                      order -- the fixed summation order of fegnn_halo_reduce_apply."""
    parts = plan.parts
    fwd_q, fwd_x, _, _ = p2p_address_tables(plan, rank, n_layers, nl_max, base_q, base_x, base_q, base_x,
                                            row_bytes_q, row_bytes_x)
    hg = parts[rank]["halo"]
    own = plan.owner[hg].astype(np.int64)
    rc = parts[rank]["recv_counts"]
    seg_start = np.concatenate([[0], np.cumsum(rc)[:-1]])                   # my halo rows are grouped by owner rank
    t = np.arange(hg.size, dtype=np.int64) - seg_start[own] if hg.size else np.zeros(0, np.int64)
    # owner o's send entries are grouped by destination d: offset of destination `rank` = sum_{d < rank} send_counts_o[d]
    send_off = np.array([int(parts[o]["send_counts"][:rank].sum()) for o in range(plan.world)], dtype=np.int64)
    slot = send_off[own] + t if hg.size else np.zeros(0, np.int64)
    brq, brx = np.asarray(base_rq, dtype=np.int64)[own], np.asarray(base_rx, dtype=np.int64)[own]
    bwd_q = [brq + (par * recv_cap + slot) * row_bytes_q for par in range(2)]
    bwd_x = [brx + (par * recv_cap + slot) * row_bytes_x for par in range(2)]
    send_idx = parts[rank]["send_idx"]
    order = np.argsort(send_idx, kind="stable")                             # by row, ties keep (user rank, halo order)
    rows, first = np.unique(send_idx[order], return_index=True)
    ptr = np.concatenate([first, [send_idx.size]]).astype(np.int64)
    return fwd_q, fwd_x, bwd_q, bwd_x, rows.astype(np.int64), ptr, order.astype(np.int64)


class FusedHaloComm(HaloComm):
    """Every exchange of the partitioned layer as ONE kernel over peer memory (csrc/halo.cu, second generation): payload
    stores into the peers' symmetric arrays, then signal / wait on per-rank signal pads inside the same kernel -- no NCCL
    call, no separate barrier launch, nothing the host has to order, so the whole partitioned training step can be one
    CUDA graph.
        forward   fegnn_halo_push_signal: owners' (Q_j, x_j) -> users' halo rows of this layer's symmetric Q / x;
                  fegnn_p2p_allreduce:    (Dsum, Usum, xsum') per layer, one-shot over symmetric slots, rank-ordered sum
        backward  fegnn_halo_push_signal: users' (dQ_j, dx_j) halo rows -> the owner's receive slots (plain stores);
                  fegnn_halo_reduce_apply: owners add their slots in fixed (rank, row) order -- DETERMINISTIC, no atomics;
                  fegnn_p2p_allreduce:    (dG1, dZ) per layer.
    Only the per-step weight-gradient all-reduce (1.3-1.7 MB) stays on NCCL."""

    AR_CAPACITY = 8192            # floats per rank and slot set: (3C + HC + 3) B <= 8192 covers C = 16 up to B = 7

    def __init__(self, plan, rank: int, device, n_layers: int, group=None):
        super().__init__(plan, rank, device, group)
        import torch.distributed._symmetric_memory as symm
        grp = dist.group.WORLD if group is None else group
        parts, W = plan.parts, plan.world
        if W > L.P2P_MAX_WORLD:
            raise L.FegnnError(f"fused halo transport supports up to {L.P2P_MAX_WORLD} ranks")
        self.n_layers = n_layers
        self.Nl_max = Nm = max(int(p["n_own"] + p["halo"].size) for p in parts)
        self.recv_cap = cap = max(1, max(int(np.sum(p["send_counts"])) for p in parts))
        f32 = dict(dtype=torch.float32, device=device)
        self.Qs, self.xs = symm.empty(n_layers, Nm, L.H, **f32), symm.empty(n_layers, Nm, 3, **f32)
        self.rq, self.rx = symm.empty(2, cap, L.H, **f32), symm.empty(2, cap, 3, **f32)
        self.ar = symm.empty(2, W, self.AR_CAPACITY, **f32)
        self.sig = symm.empty(L.P2P_CHANNELS, L.P2P_MAX_WORLD, dtype=torch.int32, device=device)
        for t in (self.Qs, self.xs, self.rq, self.rx, self.ar, self.sig):
            t.zero_()
        self.hQ, self.hx = symm.rendezvous(self.Qs, grp), symm.rendezvous(self.xs, grp)
        self.hrq, self.hrx = symm.rendezvous(self.rq, grp), symm.rendezvous(self.rx, grp)
        self.har, self.hsig = symm.rendezvous(self.ar, grp), symm.rendezvous(self.sig, grp)
        self.epoch = torch.zeros(L.P2P_CHANNELS, dtype=torch.int32, device=device)
        self.done = torch.zeros(L.P2P_CHANNELS, dtype=torch.int32, device=device)
        self.err = torch.zeros(1, dtype=torch.int32, device=device)
        self.p2p = L.P2P()
        for r in range(W):
            self.p2p.sig_peer[r] = int(self.hsig.buffer_ptrs[r])
            self.p2p.ar_peer[r] = int(self.har.buffer_ptrs[r])
        self.p2p.epoch, self.p2p.done, self.p2p.err = self.epoch.data_ptr(), self.done.data_ptr(), self.err.data_ptr()
        self.p2p.rank, self.p2p.world, self.p2p.ar_capacity = rank, W, self.AR_CAPACITY
        i64 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int64)).to(device)
        i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(device)
        fq, fx, bq, bx, rows, ptr, slots = fused_halo_tables(plan, rank, n_layers, Nm, cap, self.hQ.buffer_ptrs,
                                                             self.hx.buffer_ptrs, self.hrq.buffer_ptrs,
                                                             self.hrx.buffer_ptrs)
        self.send_idx32 = self.send_idx.to(torch.int32)
        self.fwd_q, self.fwd_x = [i64(a) for a in fq], [i64(a) for a in fx]
        self.bwd_q, self.bwd_x = [i64(a) for a in bq], [i64(a) for a in bx]
        self.b_rows, self.b_ptr, self.b_slots = i32(rows), i32(ptr), i32(slots)
        self._par = 0
        self._layer_of = {}
        torch.cuda.synchronize(device)
        dist.barrier(group=group)             # every rank has zeroed its pads / slots before anyone signals

    def check(self) -> None:
        """Host-side check of the sticky error word (a bounded wait timed out); synchronises."""
        e = int(self.err.item())
        if e:
            raise L.FegnnError(f"peer-memory exchange timed out on channel {e - 1} (a rank did not arrive)")

    # -- small all-reduces: one-shot over symmetric slots
    def allreduce(self, *tensors: torch.Tensor) -> None:
        tot = sum(t.numel() for t in tensors)
        if tot > self.AR_CAPACITY or len(tensors) > 4 or any(not t.is_contiguous() for t in tensors):
            return super().allreduce(*tensors)
        n = len(tensors)
        ptrs = (C.c_void_p * n)(*[t.data_ptr() for t in tensors])
        cnts = (C.c_int32 * n)(*[t.numel() for t in tensors])
        L.check(lib.fegnn_p2p_allreduce(C.byref(self.p2p), 2, n, ptrs, cnts, _stream(self.device)), "fegnn_p2p_allreduce")

    # -- forward
    def bind_layer(self, ph: LayerPhases, layer: int) -> None:
        ph.saved.c.Q = self.Qs[layer].data_ptr()
        self._layer_of[id(ph)] = layer

    def layer_x(self, layer: int, x: torch.Tensor, rows: int) -> torch.Tensor:
        xs = self.xs[layer, :self.Nl]
        xs[:rows].copy_(x[:rows])
        return xs

    def after_node_pre(self, ph: LayerPhases, x: torch.Tensor) -> None:
        l = self._layer_of[id(ph)]
        L.check(lib.fegnn_halo_push_signal(C.byref(self.p2p), 0, self.n_send, L.ptr(self.send_idx32), 0,
                                           L.ptr(self.fwd_q[l]), L.ptr(self.fwd_x[l]), L.ptr(self.Qs[l]), L.ptr(x),
                                           _stream(self.device)), "fegnn_halo_push_signal")

    # -- backward
    def after_edge_backward(self, ph: LayerPhases, gQ, gx, gG1, gZ_part) -> None:
        par = self._par
        self._par ^= 1
        st = _stream(self.device)
        L.check(lib.fegnn_halo_push_signal(C.byref(self.p2p), 1, self.n_recv, None, self.N, L.ptr(self.bwd_q[par]),
                                           L.ptr(self.bwd_x[par]), L.ptr(gQ), L.ptr(gx), st), "fegnn_halo_push_signal")
        L.check(lib.fegnn_halo_reduce_apply(int(self.b_rows.numel()), L.ptr(self.b_rows), L.ptr(self.b_ptr),
                                            L.ptr(self.b_slots), L.ptr(self.rq[par]), L.ptr(self.rx[par]), L.ptr(gQ),
                                            L.ptr(gx), st), "fegnn_halo_reduce_apply")
        self.allreduce(gG1, gZ_part)


# ------------------------------------------------------------------------------------- autograd driver
class _PartitionedStackFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, runner: "PartitionedFastEGNN", graph: CsrGraph, node_feat, x0, v, loc_mean, *params):
        with _on(x0.device):                  # the C ABI launches on the runtime's current device
            return _PartitionedStackFn._forward(ctx, runner, graph, node_feat, x0, v, loc_mean, *params)

    @staticmethod
    def backward(ctx, gx_out, gZ_out):
        L.deterministic("PartitionedFastEGNN backward", "multi-GPU runs are not covered, and " + L.NO_DET_LAYERS)
        with _on(ctx.saved_tensors[1].device):
            return _PartitionedStackFn._backward(ctx, gx_out, gZ_out)

    @staticmethod
    def _forward(ctx, runner: "PartitionedFastEGNN", graph: CsrGraph, node_feat, x0, v, loc_mean, *params):
        mod, comm = runner.model, runner.comm
        dev = x0.device
        N, Nl, B, Cc, Lyr = comm.N, comm.Nl, graph.B, mod.virtual_channels, mod.n_layers
        st = _stream()
        named = dict(mod.named_parameters())
        h = torch.empty(N, L.H, device=dev, dtype=torch.float32)
        L.check(lib.fegnn_embed_forward(N, node_feat.size(1), L.ptr(node_feat), L.ptr(mod.embedding_in.weight),
                                        L.ptr(mod.embedding_in.bias), L.ptr(h), st), "embed_forward")
        S = mod.virtual_node_feat.detach()[0].t().contiguous().unsqueeze(0).repeat(B, 1, 1).contiguous()
        Z = loc_mean
        p2p = isinstance(comm, (P2PHaloComm, FusedHaloComm))
        if runner._pending and p2p:
            # the saved Q / x of every layer live in per-layer symmetric arrays that a second forward would overwrite
            raise L.FegnnError("PartitionedFastEGNN: a forward started while the previous forward still waits for its "
                               "backward (peer-memory halo arrays are single-buffered per layer)")
        runner._pending = torch.is_grad_enabled()
        if isinstance(comm, P2PHaloComm):
            comm.barrier()                                                 # peers are done reading last step's arrays
        x = x0.clone()                                                     # [Nl,3]; halo rows refreshed every layer
        xsum = torch.empty(B, 3, device=dev, dtype=torch.float32)
        L.check(lib.fegnn_graph_xsum(N, B, L.ptr(x), L.ptr(graph.batch), L.ptr(xsum), st), "graph_xsum")
        comm.allreduce(xsum)
        phases, states = [], []
        for l in range(Lyr):
            flags = mod._flag_word | (L.F_LAST if l == Lyr - 1 else 0)
            dims = make_dims(N, Nl, graph.E, B, Cc, graph.Fe, flags, mod._gravity)
            ph = LayerPhases(dims, graph, layer_ptrs(named, "gcl_%d" % l), dev)
            if p2p:
                comm.bind_layer(ph, l)
                x = comm.layer_x(l, x, Nl if l == 0 else N)
            states.append((h, x, Z, S))
            h_new, x_new, Z_new, S_new, xsum = ph.forward(h, x, v, Z, S, xsum, hooks=comm)
            phases.append(ph)
            h, x, Z, S = h_new, x_new, Z_new, S_new
        ctx.runner, ctx.graph, ctx.phases, ctx.states = runner, graph, phases, states
        ctx.save_for_backward(node_feat, v)
        ctx.names = list(named.keys())
        return x[:N].contiguous(), Z

    @staticmethod
    def _backward(ctx, gx_out, gZ_out):
        runner, graph, phases, states = ctx.runner, ctx.graph, ctx.phases, ctx.states
        runner._pending = False
        mod, comm = runner.model, runner.comm
        node_feat, v = ctx.saved_tensors
        dev = v.device
        N, Nl, B, Cc, Lyr = comm.N, comm.Nl, graph.B, mod.virtual_channels, mod.n_layers
        st = _stream()
        rank0 = runner.rank == 0
        named = dict(mod.named_parameters())
        views = {n: torch.zeros_like(p) for n, p in named.items()}
        null_grads = L.LayerPtrs()                                        # replicated phases: weight grads on rank 0 only
        gZ_new = torch.zeros(B, 3, Cc, device=dev) if gZ_out is None else gZ_out.contiguous().float().clone()
        comm.allreduce(gZ_new)                                            # total dL/dZ (loss = sum of rank-local losses)
        gx_new = torch.zeros(Nl, 3, device=dev)
        if gx_out is not None:
            gx_new[:N] = gx_out
        gh = torch.zeros(N, L.H, device=dev)
        gS_new, gxsum_next = None, None
        for l in range(Lyr - 1, -1, -1):
            ph = phases[l]
            h, x, Z, S = states[l]
            live = {k: t for k, t in views.items() if k not in mod._dead_names}
            grads = layer_ptrs(live, "gcl_%d" % l)
            gh, gx_new, gZ_new, gS_new, gxsum_next = ph.backward(
                grads, h, x, v, Z, S, gh, gx_new, gZ_new, gS_new, gxsum_next, hooks=comm,
                graph_grads=grads if rank0 else null_grads)
        g_x0 = gx_new[:N] + gxsum_next[graph.batch.long()]
        g_nf = torch.empty_like(node_feat) if node_feat.requires_grad else None
        L.check(lib.fegnn_embed_backward(N, node_feat.size(1), L.ptr(node_feat), L.ptr(mod.embedding_in.weight),
                                         L.ptr(gh), L.ptr(views["embedding_in.weight"]),
                                         L.ptr(views["embedding_in.bias"]), L.ptr(g_nf), st), "embed_backward")
        if rank0:
            views["virtual_node_feat"].copy_(gS_new.sum(0).t().unsqueeze(0))
        runner.last_local_grads = views
        grads_out = tuple(None if n in mod._dead_names else views[n] for n in ctx.names)
        g_x0_full = torch.zeros(Nl, 3, device=dev)
        g_x0_full[:N] = g_x0
        return (None, None, g_nf, g_x0_full, None, gZ_new) + grads_out


class PartitionedFastEGNN:
    """Runs a FastEGNN module (same weights on every rank) on this rank's slab of one big graph."""

    def __init__(self, model, plan: SlabPlan, rank: int, device, group=None, halo: str = "nccl"):
        """halo = "nccl": pack + all-to-all + unpack; "p2p": direct peer stores / remote atomics over NVLink
        (P2PHaloComm; needs torch symmetric memory, i.e. all ranks on one NVLink / NVSwitch domain)."""
        if getattr(model, "_node_attr_nf", 0) != 0:
            raise NotImplementedError("the partitioned path has no node attributes: build the model with node_attr_nf=0")
        self.model, self.plan, self.rank = model, plan, rank
        if halo == "fused":
            self.comm = FusedHaloComm(plan, rank, device, model.n_layers, group)
        elif halo == "p2p":
            self.comm = P2PHaloComm(plan, rank, device, model.n_layers, group)
        elif halo == "nccl":
            self.comm = HaloComm(plan, rank, device, group)
        else:
            raise ValueError(f"halo must be 'nccl', 'p2p' or 'fused', got {halo!r}")
        self.last_local_grads = None
        self._pending = False
        self._flat = None

    def __call__(self, node_feat, node_loc, node_vel, edge_index, loc_mean, edge_attr, n_global: int):
        """node_* hold this rank's owned rows followed by its halo rows ([Nl, .]); edge_index is local
        (row < N owned, col < Nl) -- or this rank's prebuilt CsrGraph (DeviceSlabPlan.graph; edge_attr must then be None);
        loc_mean [1,3,C] is replicated.  Returns (x' of the OWNED rows, Z')."""
        L.deterministic("PartitionedFastEGNN", "multi-GPU runs are not covered, and " + L.NO_DET_LAYERS)
        _require_cuda(node_loc, "node_loc")
        N = self.comm.N
        B = int(loc_mean.size(0))
        if B != 1:
            raise L.FegnnError(f"the partitioned path runs ONE graph across the ranks (loc_mean has B={B}); batches of "
                               "small graphs go whole to the ranks (data parallel)")
        if isinstance(edge_index, CsrGraph):
            graph = edge_index
            if edge_attr is not None:
                raise TypeError("edge_attr must be None when edge_index is a prebuilt CsrGraph (it carries its own)")
            if graph.live:
                raise L.FegnnError("the partitioned runner takes graphs with a host-known edge count: a live graph "
                                   "(CsrGraph.from_radius(capacity=...) or CsrGraph(..., n_edges=...)) is not supported here")
            if graph.N != N or graph.Nl != self.comm.Nl:
                raise L.FegnnError(f"prebuilt slab graph (N={graph.N}, Nl={graph.Nl}) does not match the plan "
                                   f"(N={N}, Nl={self.comm.Nl})")
        else:
            batch = torch.zeros(N, dtype=torch.int64, device=node_loc.device)
            graph = CsrGraph(edge_index, batch, edge_attr, B, n_local=self.comm.Nl)
            graph.inv_nb.fill_(1.0 / max(1, n_global))                    # graph size is global, not the slab's
        params = [p for _, p in self.model.named_parameters()]
        with _on(node_loc.device):
            return _PartitionedStackFn.apply(self, graph, node_feat[:N].contiguous().float(),
                                             node_loc.contiguous().float(), node_vel[:N].contiguous().float(),
                                             loc_mean.contiguous().float(), *params)

    def allreduce_gradients(self) -> None:
        """Sum the weight gradients over ranks (one collective on a flat buffer)."""
        grads = [p.grad for p in self.model.parameters() if p.grad is not None]
        bases = {(g._base if g._base is not None else g).data_ptr() for g in grads}
        if len(bases) == 1 and grads[0]._base is not None and grads[0]._base.is_contiguous():
            dist.all_reduce(grads[0]._base, group=self.comm.group)      # the gradients are views of one flat buffer
            return
        flat = torch._utils._flatten_dense_tensors(grads)
        dist.all_reduce(flat, group=self.comm.group)
        torch._foreach_copy_(grads, list(torch._utils._unflatten_dense_tensors(flat, grads)))
