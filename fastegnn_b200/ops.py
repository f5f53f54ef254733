"""Thin host wrappers over the C ABI: graph prep, per-layer pointer tables, the MMD op.

Everything here is plumbing (device buffers from torch, raw pointers into libfegnn.so);
no arithmetic of the path is done in Python.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import torch

from . import _lib as L

lib = L.lib


def _stream(dev=None):
    """cudaStream_t of torch's current stream ON THE TENSORS' DEVICE (not the thread's current device: the reference mains
    take --device cuda:N without torch.cuda.set_device)."""
    return torch.cuda.current_stream(dev).cuda_stream


def _on(dev):
    """Device guard for a C-ABI call: libfegnn launches on the CUDA runtime's current device."""
    return torch.cuda.device(dev)


def _require_cuda(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise L.FegnnError(
            f"{name} is on {t.device}: fastegnn_b200 runs on CUDA (sm_100a) only and has no CPU fallback")


_PREP_STREAMS = {}


def _prep_stream(dev) -> "torch.cuda.Stream":
    """One side stream per device for CsrGraph(overlap=True)."""
    key = torch.device(dev).index if torch.device(dev).index is not None else torch.cuda.current_device()
    if key not in _PREP_STREAMS:
        _PREP_STREAMS[key] = torch.cuda.Stream(device=key)
    return _PREP_STREAMS[key]


class CsrGraph:
    """CSR-by-row view of one batch (output of fegnn_graph_prep), shared by all layers
    and by backward.  Replaces the per-layer int64 gathers / scatter_add of
    models/FastEGNN.py:182,210,279-294."""

    def __init__(self, edge_index: torch.Tensor, data_batch: torch.Tensor, edge_attr: Optional[torch.Tensor],
                 n_graphs: int, n_local: Optional[int] = None, overlap: bool = False):
        """overlap=True runs the sort on a per-device side stream and leaves `ready_event` in the pointer table:
        fegnn_model_forward joins it right before its first use of the CSR arrays (the embedding and the first layer's
        node phase run under the sort).  Any other consumer must call wait() first."""
        _require_cuda(edge_index, "edge_index")
        dev = edge_index.device
        N = int(data_batch.numel())
        E = int(edge_index.size(1))
        Fe = 0 if edge_attr is None else int(edge_attr.size(1))
        if edge_index.dtype != torch.int64 or data_batch.dtype != torch.int64:
            raise L.FegnnError("edge_index / data_batch must be int64 (as produced by the reference loaders)")
        ei = edge_index.contiguous()
        db = data_batch.contiguous()
        ea = None if edge_attr is None else edge_attr.contiguous().float()
        self.N, self.E, self.B, self.Fe = N, E, n_graphs, Fe
        self.Nl = N if n_local is None else n_local
        i32 = dict(device=dev, dtype=torch.int32)
        f32 = dict(device=dev, dtype=torch.float32)
        self.perm = torch.empty(E, **i32)
        self.rowptr = torch.empty(N + 1, **i32)
        self.row = torch.empty(E, **i32)
        self.col = torch.empty(E, **i32)
        self.batch = torch.empty(N, **i32)
        self.gptr = torch.empty(n_graphs + 1, **i32)
        self.edge_attr = torch.empty(E, max(Fe, 1), **f32) if Fe else torch.empty(0, **f32)
        self.dinv = torch.empty(N, **f32)
        self.inv_nb = torch.empty(n_graphs, **f32)
        nbytes = int(lib.fegnn_graph_prep_workspace_bytes(N, E))
        ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
        self._ready = None
        with _on(dev):
            # every buffer above was allocated under the caller's stream; with overlap the side stream first joins that
            # stream (inputs and recycled memory are ordered), then runs the sort while the caller's stream goes on
            main = torch.cuda.current_stream(dev)
            st = main
            if overlap:
                st = _prep_stream(dev)
                st.wait_stream(main)
            L.check(lib.fegnn_graph_prep(N, E, n_graphs, Fe, L.ptr(ei), L.ptr(db), L.ptr(ea), L.ptr(self.perm),
                                         L.ptr(self.rowptr), L.ptr(self.row), L.ptr(self.col), L.ptr(self.batch),
                                         L.ptr(self.gptr), L.ptr(self.edge_attr), L.ptr(self.dinv), L.ptr(self.inv_nb),
                                         L.ptr(ws), nbytes, st.cuda_stream), "fegnn_graph_prep")
            if overlap:
                self._ready = torch.cuda.Event()
                self._ready.record(st)
        self._ws = ws   # stream-ordered: keep alive until the kernels that use it have been enqueued
        self._keep = (ei, db, ea)   # inputs of a sort that may still be running on the side stream
        self.rebind()

    def rebind(self) -> None:
        """(Re)build the fegnn_graph pointer table from the current tensors (after slicing / renumbering them)."""
        ready = getattr(self, "_ready", None)
        self.c = L.Graph(L.ptr(self.row), L.ptr(self.col), L.ptr(self.batch), L.ptr(self.edge_attr),
                         L.ptr(self.dinv), L.ptr(self.inv_nb), None if ready is None else ready.cuda_event)

    def wait(self) -> None:
        """Order the current stream behind a sort that runs on the side stream (no-op otherwise)."""
        ready = getattr(self, "_ready", None)
        if ready is not None:
            torch.cuda.current_stream(self.row.device).wait_event(ready)
            self._ready = None
            self.c.ready_event = None

    @classmethod
    def from_radius(cls, node_loc: torch.Tensor, data_batch: torch.Tensor, n_graphs: int, r: float,
                    cutoff_rate: float = 0.0, edge_attr_nf: int = 2) -> "CsrGraph":
        """Build the graph ON THE DEVICE (fegnn_radius_graph_count / _fill): every ordered pair of distinct nodes of
        the same graph closer than r, the shortest int(E_b (1 - cutoff_rate)) of them per graph, in CSR order with
        edge_attr = length in each of the edge_attr_nf columns.  Replaces radius_graph + cutoff_edge + norm of
        datasets/simulation/dataset.py:80-82,96-101 (r = math.inf: the complete-graph / topk selection of
        datasets/nbody/dataset.py:102-113) and the per-forward CSR sort.  One host read of the candidate count
        sizes the buffers (this is dataset-time work, not part of the captured training step)."""
        _require_cuda(node_loc, "node_loc")
        dev = node_loc.device
        x = node_loc.detach().contiguous().float()
        if data_batch.dtype != torch.int64:
            raise L.FegnnError("data_batch must be int64 (as produced by the reference loaders)")
        db = data_batch.contiguous()
        N, B, Fe = int(x.size(0)), int(n_graphs), int(edge_attr_nf)
        if not r > 0:
            raise L.FegnnError("r must be positive (math.inf for the complete graph)")
        if not 0.0 <= cutoff_rate <= 1.0:
            raise L.FegnnError("cutoff_rate must be in [0, 1]")
        i32 = dict(device=dev, dtype=torch.int32)
        f32 = dict(device=dev, dtype=torch.float32)
        self = cls.__new__(cls)
        self.N, self.B, self.Fe, self.Nl = N, B, Fe, N
        self.perm = None                                      # there is no caller-side edge list to permute
        self.batch = torch.empty(N, **i32)
        self.gptr = torch.empty(B + 1, **i32)
        self.inv_nb = torch.empty(B, **f32)
        self.dinv = torch.empty(N, **f32)
        self.rowptr = torch.empty(N + 1, **i32)
        cand_rowptr = torch.empty(N + 1, **i32)
        counts = torch.zeros(2, **i32)                        # [n_cand, n_edges]
        nbytes = int(lib.fegnn_radius_graph_workspace_bytes(N, B))
        ws = torch.empty(nbytes, device=dev, dtype=torch.uint8)
        st = _stream(dev)
        with _on(dev):
            L.check(lib.fegnn_radius_graph_count(N, B, L.ptr(x), L.ptr(db), float(r), L.ptr(self.batch), L.ptr(self.gptr),
                                                 L.ptr(self.inv_nb), L.ptr(cand_rowptr), L.ptr(counts[0:1]), L.ptr(ws),
                                                 nbytes, st), "fegnn_radius_graph_count")
        n_cand = int(counts[0].item())
        keep_frac = 1.0 - float(cutoff_rate)                  # the reference's int(E * (1 - cutoff_rate)) in fp64
        cap = max(n_cand, 1)
        ccol = torch.empty(cap, **i32)
        crow = torch.empty(cap, **i32)
        cdist = torch.empty(cap, **f32)
        row = torch.empty(cap, **i32)
        col = torch.empty(cap, **i32)
        ea = torch.empty(cap, max(Fe, 1), **f32)
        with _on(dev):
            L.check(lib.fegnn_radius_graph_fill(N, B, Fe, float(r), keep_frac, L.ptr(self.batch), L.ptr(self.gptr),
                                                L.ptr(cand_rowptr), L.ptr(counts[0:1]), n_cand, L.ptr(ccol), L.ptr(cdist),
                                                L.ptr(crow), cap, L.ptr(self.rowptr), L.ptr(row), L.ptr(col), L.ptr(ea),
                                                L.ptr(self.dinv), L.ptr(counts[1:2]), L.ptr(ws), nbytes, st),
                    "fegnn_radius_graph_fill")
        E = int(counts[1].item())
        self.E = E
        self.n_candidates = n_cand
        self.row, self.col = row[:E], col[:E]
        self.edge_attr = ea[:E] if Fe else torch.empty(0, **f32)
        self._ws = ws
        self.rebind()
        return self

    def edge_index(self) -> torch.Tensor:
        """int64 [2,E] view of the CSR edge list for callers that want the reference's tensor (a cast, no arithmetic)."""
        return torch.stack([self.row.long(), self.col.long()])


def make_dims(N: int, Nl: int, E: int, B: int, C_: int, Fe: int, flags: int,
              gravity: Optional[Sequence[float]] = None, eps: float = 1e-8, Fa: int = 0,
              node_attr: Optional[torch.Tensor] = None) -> L.Dims:
    """fegnn_dims.  node_attr: [N, Fa] fp32 tensor (kept alive by the caller while the dims are in use) or None."""
    d = L.Dims()
    d.N, d.Nl, d.E, d.B, d.C, d.Fe, d.flags = N, Nl, E, B, C_, Fe, flags
    g = (0.0, 0.0, 0.0) if gravity is None else tuple(float(x) for x in gravity)
    d.gravity[0], d.gravity[1], d.gravity[2] = g
    d.eps = eps
    d.Fa, d.node_attr = Fa, L.ptr(node_attr)
    return d


def node_attr_arg(node_attr, node_attr_nf: int, n_nodes: int) -> Optional[torch.Tensor]:
    """Checks the node_attr argument of a forward against the module's node_attr_nf (before any device work, as
    edge_attr is checked) and returns it as a contiguous fp32 CUDA tensor, or None when the module takes none."""
    if node_attr is None:
        if node_attr_nf != 0:
            raise TypeError(f"node_attr is required when node_attr_nf > 0 (got None, node_attr_nf={node_attr_nf}; the "
                            "reference's torch.cat fails on None, models/FastEGNN.py:159)")
        return None
    if node_attr_nf == 0:
        raise RuntimeError("node_attr was given to a model built with node_attr_nf=0")
    if node_attr.dim() != 2 or node_attr.size(1) != node_attr_nf:
        raise RuntimeError(f"node_attr has shape {tuple(node_attr.shape)}, model was built with node_attr_nf={node_attr_nf}")
    if node_attr.size(0) != n_nodes:
        raise RuntimeError(f"node_attr has {node_attr.size(0)} rows for {n_nodes} nodes")
    _require_cuda(node_attr, "node_attr")
    return node_attr.detach().contiguous().float()


def layer_ptrs(tensors: Dict[str, torch.Tensor], prefix: str) -> L.LayerPtrs:
    """Pointer table of one layer from reference-named tensors (missing names -> NULL)."""
    p = L.LayerPtrs()
    for field, suffix in L.LAYER_FIELDS:
        t = tensors.get(f"{prefix}.{suffix}" if prefix else suffix)
        if t is not None:
            if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
                raise L.FegnnError(f"parameter {prefix}.{suffix} must be a contiguous fp32 CUDA tensor")
            setattr(p, field, t.data_ptr())
    return p


class SavedBlock:
    """One layer's kept activations: a flat buffer carved by fegnn_layer_saved_bind."""

    def __init__(self, dims: L.Dims, device):
        n = int(lib.fegnn_layer_saved_floats(C.byref(dims)))
        self.buf = torch.empty(n, device=device, dtype=torch.float32)
        self.c = L.Saved()
        L.check(lib.fegnn_layer_saved_bind(C.byref(dims), L.ptr(self.buf), C.byref(self.c)), "fegnn_layer_saved_bind")
        self.dims = dims

    def view(self, name: str, shape) -> torch.Tensor:
        off = (getattr(self.c, name) - self.buf.data_ptr()) // 4
        n = 1
        for s in shape:
            n *= s
        return self.buf[off:off + n].view(*shape)


# ----------------------------------------------------------------------------- MMD
def _loss_workspace(N: int, B: int, dev):
    """Per-CTA partials of the deterministic loss forward (None and 0 with the mode off)."""
    n = int(lib.fegnn_loss_workspace_floats(N, B))
    return (torch.empty(n, device=dev, dtype=torch.float32) if n else None), n


class _MmdFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, Z, sample_idx, sigma, scale_vv, scale_rv):
        _require_cuda(x, "node_loc")
        x = x.contiguous()
        Z = Z.contiguous()
        B, _, C_ = Z.shape
        ns = sample_idx.size(1)
        loss = torch.empty(1, device=x.device, dtype=torch.float32)
        ctx.det = L.deterministic("mmd_loss")
        ws, nws = _loss_workspace(0, B, x.device)
        with _on(x.device):
            L.check(lib.fegnn_mmd_forward(B, C_, ns, float(sigma), float(scale_vv), float(scale_rv), L.ptr(x), L.ptr(Z),
                                          L.ptr(sample_idx), L.ptr(loss), L.ptr(ws), nws, _stream(x.device)),
                    "fegnn_mmd_forward")
        ctx.save_for_backward(x, Z, sample_idx)
        ctx.cfg = (float(sigma), float(scale_vv), float(scale_rv))
        return loss[0]

    @staticmethod
    def backward(ctx, g):
        x, Z, idx = ctx.saved_tensors
        B, _, C_ = Z.shape
        sigma, svv, srv = ctx.cfg
        gx = torch.empty_like(x)
        gZ = torch.empty_like(Z)
        gl = g.reshape(1).contiguous().float()
        L.set_mode("deterministic", int(ctx.det))          # the backward takes the summation order of its forward
        with _on(x.device):
            L.check(lib.fegnn_mmd_backward(x.size(0), B, C_, idx.size(1), sigma, svv, srv, L.ptr(x), L.ptr(Z), L.ptr(idx),
                                           L.ptr(gl), L.ptr(gx), L.ptr(gZ), _stream(x.device)), "fegnn_mmd_backward")
        return gx, gZ, None, None, None, None


def mmd_loss(node_loc: torch.Tensor, virtual_node_loc: torch.Tensor, sample_idx: torch.Tensor, sigma: float,
             scale_vv: float = 1.0, scale_rv: float = 1.0):
    """l_vv - l_rv of utils/train.py:111-165 in one launch.

    node_loc [N,3]; virtual_node_loc [B,3,C] exactly as FastEGNN.forward returns it (the
    reference permutes it to [B,C,3] at :113); sample_idx int32 [B, ns] of GLOBAL node
    indices (graph offset + the reference's torch.randperm(n_b)[:ns]).  scale_vv / scale_rv weight the two terms (1, 1 =
    the reference; the partitioned path splits the sum over ranks, see fegnn.h).  Under
    torch.use_deterministic_algorithms(True) the result and its gradients are bitwise reproducible as long as no node
    index appears in the samples of two different graphs (true when each graph samples its own nodes)."""
    if sample_idx.dtype != torch.int32:
        sample_idx = sample_idx.to(torch.int32)
    return _MmdFn.apply(node_loc, virtual_node_loc, sample_idx.contiguous(), sigma, scale_vv, scale_rv)


class _MseMmdFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, target, Z, sample_idx, sigma, weight, scale_vv, scale_rv, inv_count):
        _require_cuda(x, "node_loc")
        x, target, Z = x.contiguous(), target.contiguous().float(), Z.contiguous()
        B, _, C_ = Z.shape
        total = torch.empty((), device=x.device, dtype=torch.float32)
        mse = torch.empty((), device=x.device, dtype=torch.float32)
        ctx.det = L.deterministic("mse_mmd_loss")
        ws, nws = _loss_workspace(x.size(0), B, x.device)
        with _on(x.device):
            L.check(lib.fegnn_mse_mmd_forward(x.size(0), B, C_, sample_idx.size(1), float(sigma), float(weight),
                                              float(scale_vv), float(scale_rv), float(inv_count), L.ptr(x), L.ptr(target),
                                              L.ptr(Z), L.ptr(sample_idx), L.ptr(total), L.ptr(mse), L.ptr(ws), nws,
                                              _stream(x.device)),
                    "fegnn_mse_mmd_forward")
        ctx.save_for_backward(x, target, Z, sample_idx)
        ctx.cfg = (float(sigma), float(weight), float(scale_vv), float(scale_rv), float(inv_count))
        ctx.set_materialize_grads(False)         # an unused output arrives as None in backward, not as a zero-fill kernel
        return total, mse

    @staticmethod
    def backward(ctx, g_total, g_mse):
        x, target, Z, idx = ctx.saved_tensors
        B, _, C_ = Z.shape
        sigma, weight, svv, srv, inv_count = ctx.cfg
        gx = torch.empty_like(x)
        gZ = torch.empty_like(Z)
        gt = None if g_total is None else g_total.reshape(1).contiguous().float()
        gm = None if g_mse is None else g_mse.reshape(1).contiguous().float()
        L.set_mode("deterministic", int(ctx.det))
        with _on(x.device):
            L.check(lib.fegnn_mse_mmd_backward(x.size(0), B, C_, idx.size(1), sigma, weight, svv, srv, inv_count, L.ptr(x),
                                               L.ptr(target), L.ptr(Z), L.ptr(idx), L.ptr(gt), L.ptr(gm), L.ptr(gx), L.ptr(gZ),
                                               _stream(x.device)), "fegnn_mse_mmd_backward")
        return gx, None, gZ, None, None, None, None, None, None


def mse_mmd_loss(node_loc: torch.Tensor, target: torch.Tensor, virtual_node_loc: torch.Tensor, sample_idx: torch.Tensor,
                 sigma: float, weight: float, scale_vv: float = 1.0, scale_rv: float = 1.0, inv_count: float = None):
    """The training step's loss of utils/train.py:104-163 in one launch per direction:
    `total = mse_loss(node_loc, target) + weight * mmd_loss(node_loc, virtual_node_loc, sample_idx, sigma)`.
    Returns (total, mse): `total` is what the loop back-propagates (:166), `mse` what it logs (:107).  No gradient flows to
    `target`.  inv_count defaults to 1 / node_loc.numel() (torch's mean reduction).  Deterministic under
    torch.use_deterministic_algorithms(True) on the same condition as mmd_loss."""
    if sample_idx.dtype != torch.int32:
        sample_idx = sample_idx.to(torch.int32)
    if inv_count is None:
        inv_count = 1.0 / max(1, node_loc.numel())
    total, mse = _MseMmdFn.apply(node_loc, target, virtual_node_loc, sample_idx.contiguous(), sigma, weight, scale_vv,
                                 scale_rv, inv_count)
    return total, mse


# ----------------------------------------------------------------------------- unsorted_segment_sum / _mean
class _SegmentFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, data, ids, num_segments, mean):
        _require_cuda(data, "data")
        dev = data.device
        if ids.dtype != torch.int64:
            raise L.FegnnError("segment_ids must be int64 (as in the reference)")
        d2 = data.contiguous().float()
        E, K = int(d2.size(0)), int(d2.size(1))
        ids = ids.contiguous()
        out = torch.empty(num_segments, K, device=dev, dtype=torch.float32)
        cnt = torch.empty(num_segments, device=dev, dtype=torch.float32) if mean else None
        with _on(dev):
            L.check(lib.fegnn_segment_reduce(E, K, int(num_segments), L.ptr(d2), L.ptr(ids), int(bool(mean)), L.ptr(out),
                                             L.ptr(cnt), _stream(dev)), "fegnn_segment_reduce")
        ctx.save_for_backward(ids, cnt) if mean else ctx.save_for_backward(ids)
        ctx.cfg = (E, K, int(num_segments), bool(mean))
        return out

    @staticmethod
    def backward(ctx, g):
        E, K, S, mean = ctx.cfg
        ids = ctx.saved_tensors[0]
        cnt = ctx.saved_tensors[1] if mean else None
        g = g.contiguous().float()
        gd = torch.empty(E, K, device=g.device, dtype=torch.float32)
        with _on(g.device):
            L.check(lib.fegnn_segment_reduce_backward(E, K, S, L.ptr(g), L.ptr(ids), L.ptr(cnt), L.ptr(gd),
                                                      _stream(g.device)), "fegnn_segment_reduce_backward")
        return gd, None, None, None


def segment_reduce(data: torch.Tensor, segment_ids: torch.Tensor, num_segments: int, mean: bool) -> torch.Tensor:
    """unsorted_segment_sum / unsorted_segment_mean of models/FastEGNN.py:279-294 (2-D data, int64 ids)."""
    L.deterministic("unsorted_segment_mean" if mean else "unsorted_segment_sum", "a scatter by segment id with float atomics")
    return _SegmentFn.apply(data, segment_ids, int(num_segments), bool(mean))
