"""One E_GCL_vel layer driven phase by phase through the C ABI (models/FastEGNN.py:192-223).

`FastEGNN.forward` uses the two whole-stack C calls; this module is the layer-level entry
point (`E_GCL_vel.forward`, the unit the "layer fwd+bwd edges/s" metric is quoted on) and
the building block of the spatially partitioned multi-GPU path, which needs to exchange
halo rows and all-reduce per-graph sums BETWEEN phases (fastegnn_b200/partitioned.py).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib as L
from .ops import CsrGraph, SavedBlock, _on, _require_cuda, _stream, layer_ptrs, live_flag, make_dims

lib = L.lib


def _f32(t):
    return t.contiguous().float()


class LayerPhases:
    """Buffers + phase calls for one layer on one device.  `hooks` lets the partitioned path
    insert communication between phases; on one GPU every hook is a no-op."""

    def __init__(self, dims: L.Dims, graph: CsrGraph, params: L.LayerPtrs, device):
        self.d, self.g, self.p, self.dev = dims, graph, params, device
        self.pd = C.byref(dims)
        self.saved = SavedBlock(dims, device)
        self.last = bool(dims.flags & L.F_LAST)

    def _e(self, *shape):
        return torch.empty(*shape, device=self.dev, dtype=torch.float32)

    # ---- forward
    def forward(self, h, x, v, Z, S, xsum, hooks=None):
        with _on(self.dev):                      # the C ABI launches on the runtime's current device
            return self._forward(h, x, v, Z, S, xsum, hooks)

    def backward(self, grads, h, x, v, Z, S, gh_new, gx_new, gZ_new, gS_new, gxsum_next, hooks=None, graph_grads=None,
                 input_grads: Optional[L.InputGrads] = None):
        with _on(self.dev):
            return self._backward(grads, h, x, v, Z, S, gh_new, gx_new, gZ_new, gS_new, gxsum_next, hooks, graph_grads,
                                  input_grads)

    def _forward(self, h, x, v, Z, S, xsum, hooks=None):
        d, g, p, sv, st = self.d, self.g, self.p, self.saved, _stream(self.dev)
        N, B, Cc = d.N, d.B, d.C
        pd, pg, pp, ps = self.pd, C.byref(g.c), C.byref(p), C.byref(sv.c)
        L.check(lib.fegnn_graph_pre_forward(pd, pg, pp, L.ptr(Z), L.ptr(S), L.ptr(xsum), ps, st), "graph_pre_forward")
        L.check(lib.fegnn_node_pre_forward(pd, pp, L.ptr(h), ps, st), "node_pre_forward")
        if hooks is not None:
            hooks.after_node_pre(self, x)            # halo exchange of Q and x
        L.check(lib.fegnn_edge_forward(pd, pg, pp, L.ptr(x), ps, st), "edge_forward")
        x_new = self._e(d.Nl, 3)
        xsum_new = self._e(B, 3)
        L.check(lib.fegnn_virtual_forward(pd, pg, pp, L.ptr(x), L.ptr(v), L.ptr(Z), ps, L.ptr(x_new),
                                          L.ptr(xsum_new), st), "virtual_forward")
        if hooks is not None:
            hooks.after_virtual(self, xsum_new)      # all-reduce of Dsum, Usum, xsum_new
        h_new = None
        if not self.last:
            h_new = self._e(N, L.H)
            L.check(lib.fegnn_node_h_forward(pd, pg, pp, L.ptr(h), ps, L.ptr(h_new), st), "node_h_forward")
        Z_new = self._e(B, 3, Cc)
        S_new = None if self.last else self._e(B, Cc, L.H)
        L.check(lib.fegnn_graph_post_forward(pd, pg, pp, L.ptr(Z), L.ptr(S), ps, L.ptr(Z_new), L.ptr(S_new), st),
                "graph_post_forward")
        return h_new, x_new, Z_new, S_new, xsum_new

    # ---- backward
    def _backward(self, grads: L.LayerPtrs, h, x, v, Z, S, gh_new, gx_new, gZ_new, gS_new, gxsum_next, hooks=None,
                  graph_grads: Optional[L.LayerPtrs] = None, input_grads: Optional[L.InputGrads] = None):
        """gh_new is consumed in place (becomes dL/dh).  Returns (gh, gx, gZ, gS, gxsum).
        graph_grads: weight-gradient table for the per-graph phases (replicated when partitioned, so
        only one rank passes real pointers); defaults to `grads`.  input_grads: buffers the phases ADD this layer's
        node_vel / node_attr / edge_attr gradients into (fegnn_input_grads), or None."""
        d, g, p, sv, st = self.d, self.g, self.p, self.saved, _stream(self.dev)
        N, Nl, B, Cc = d.N, d.Nl, d.B, d.C
        pd, pg, pp, ps, pgr = self.pd, C.byref(g.c), C.byref(p), C.byref(sv.c), C.byref(grads)
        pig = None if input_grads is None else C.byref(input_grads)
        pgg = pgr if graph_grads is None else C.byref(graph_grads)
        gZ, gS = self._e(B, 3, Cc), self._e(B, Cc, L.H)
        gDsum, gUsum = self._e(B, 3, Cc), self._e(B, Cc, L.H)
        L.check(lib.fegnn_graph_post_backward(pd, pg, pp, pgg, L.ptr(S), ps, L.ptr(gZ_new), L.ptr(gS_new), L.ptr(gZ),
                                              L.ptr(gS), L.ptr(gDsum), L.ptr(gUsum), st), "graph_post_backward")
        gzh1 = gm = None
        gu = self._e(N, Cc, L.H)      # last layer: no input (FEGNN_F_LAST), still the scratch of the tensor-core kernels
        if not self.last:
            gzh1, gm, gu = self._e(N, L.H), self._e(N, L.H), self._e(N, Cc, L.H)
            L.check(lib.fegnn_node_h_backward(pd, pg, pp, pgr, ps, L.ptr(gh_new), L.ptr(gzh1), L.ptr(gm), L.ptr(gu),
                                              st), "node_h_backward")
        gAv, gG1 = self._e(N, L.H), self._e(B, Cc, L.H)
        own_buffers = getattr(hooks, "grad_halo_buffers", None)      # peer-memory halo path: gQ / gx live in symmetric memory
        gQ, gx = own_buffers(self) if own_buffers is not None else (self._e(Nl, L.H), self._e(Nl, 3))
        gsv, gsg, gt = self._e(N), self._e(N), self._e(N, 3)
        # partitioned: the virtual phase adds only this rank's share of dZ -> keep it apart until it is all-reduced
        gZ_part = gZ if hooks is None else torch.zeros(B, 3, Cc, device=self.dev, dtype=torch.float32)
        L.check(lib.fegnn_virtual_backward_inputs(pd, pg, pp, pgr, L.ptr(x), L.ptr(v), L.ptr(Z), ps, L.ptr(gx_new),
                                                  L.ptr(gxsum_next), L.ptr(gDsum), None if self.last else L.ptr(gUsum),
                                                  L.ptr(gu), L.ptr(gAv), L.ptr(gG1), L.ptr(gx), L.ptr(gZ_part), L.ptr(gsv),
                                                  L.ptr(gsg), L.ptr(gt), pig, st), "virtual_backward")
        gP = self._e(N, L.H)
        L.check(lib.fegnn_edge_backward_inputs(pd, pg, pp, pgr, L.ptr(x), ps, L.ptr(gm), L.ptr(gt), L.ptr(gP), L.ptr(gQ),
                                               L.ptr(gx), pig, st), "edge_backward")
        if hooks is not None:
            hooks.after_edge_backward(self, gQ, gx, gG1, gZ_part)   # reverse halo (sum) + all-reduce of dG1 / dZ shares
            gZ.add_(gZ_part)
        gxsum = self._e(B, 3)
        L.check(lib.fegnn_graph_pre_backward(pd, pg, pp, pgg, L.ptr(S), ps, L.ptr(gG1), L.ptr(gS), L.ptr(gZ),
                                             L.ptr(gxsum), st), "graph_pre_backward")
        L.check(lib.fegnn_node_pre_backward_inputs(pd, pp, pgr, L.ptr(h), L.ptr(gP), L.ptr(gQ), L.ptr(gAv), L.ptr(gzh1),
                                                   L.ptr(gsv), L.ptr(gsg), L.ptr(gh_new), pig, st), "node_pre_backward")
        return gh_new, gx, gZ, gS, gxsum


def _layer_named(layer):
    return [(n, p) for n, p in layer.named_parameters()]


class _LayerFn(torch.autograd.Function):
    """One layer through the phase calls, as a function of NAMED WEIGHT TENSORS (reference state_dict suffixes, any
    autograd history): E_GCL_vel.forward passes a layer's parameters; the VNEGNN sibling passes tensors it assembles from
    its own parameters (fastegnn_b200/VNEGNN.py).  spec = (names, flag word, gravity list or None, virtual channels).
    node_attr is the fp32 copy the kernels read; attr_in / edge_attr_in are the caller's node_attr / edge_attr tensors (or
    None), inputs only so that autograd hands them their gradients (the kernels read edge_attr from the graph)."""

    @staticmethod
    def forward(ctx, spec, graph, node_attr, attr_in, edge_attr_in, h, x, v, Z, S, *params):
        names, flags, grav, Cc = spec
        L.deterministic("the FastEGNN layer", L.NO_DET_LAYERS)
        dev = x.device
        named = dict(zip(names, params))
        ptrs = layer_ptrs(named, "")
        Fa = 0 if node_attr is None else node_attr.size(1)
        # a live graph (CsrGraph.live): E is its capacity and the phases read the live count (FEGNN_F_LIVE_EDGES)
        dims = make_dims(graph.N, graph.N, graph.E, graph.B, Cc, graph.Fe, flags | live_flag(graph), grav, Fa=Fa,
                         node_attr=node_attr)
        ph = LayerPhases(dims, graph, ptrs, dev)
        xsum = torch.empty(graph.B, 3, device=dev, dtype=torch.float32)
        with _on(dev):
            L.check(lib.fegnn_graph_xsum(graph.N, graph.B, L.ptr(x), L.ptr(graph.batch), L.ptr(xsum), _stream(dev)),
                    "graph_xsum")
        h_new, x_new, Z_new, S_new, _ = ph.forward(h, x, v, Z, S, xsum)
        ctx.ph = ph
        ctx.node_attr = node_attr          # ph.d points at it until the backward
        ctx.save_for_backward(h, x, v, Z, S, *params)
        ctx.names = names
        ctx.in_dtypes = (None if attr_in is None else attr_in.dtype, None if edge_attr_in is None else edge_attr_in.dtype)
        return h_new, x_new, S_new, Z_new

    @staticmethod
    def backward(ctx, gh_new, gx_new, gS_new, gZ_new):
        ph = ctx.ph
        L.deterministic("the FastEGNN layer backward", L.NO_DET_LAYERS)
        h, x, v, Z, S = ctx.saved_tensors[:5]
        params = ctx.saved_tensors[5:]
        z = lambda t, ref: torch.zeros_like(ref) if t is None else t.contiguous().float()
        gh_new = z(gh_new, h).clone()
        gx_new, gS_new, gZ_new = z(gx_new, x), z(gS_new, S), z(gZ_new, Z)
        views = {n: torch.zeros_like(p) for n, p in zip(ctx.names, params)}
        gptrs = layer_ptrs(views, "")
        need = ctx.needs_input_grad
        zf = lambda *shape: torch.zeros(*shape, device=x.device, dtype=torch.float32)      # the phases add into these
        g_na = zf(ph.d.N, ph.d.Fa) if need[3] else None
        g_ea = zf(ph.g.E, ph.g.Fe) if need[4] else None
        g_v = zf(ph.d.N, 3) if need[7] else None
        ig = None
        if g_na is not None or g_ea is not None or g_v is not None:
            ig = L.InputGrads(L.ptr(g_v), L.ptr(g_na), L.ptr(g_ea) if ph.g.Fe else None, L.ptr(ph.g.perm))
        gh, gx, gZ, gS, gxsum = ph.backward(gptrs, h, x, v, Z, S, gh_new, gx_new, gZ_new, gS_new, None, input_grads=ig)
        gx = gx + gxsum[ph.g.batch.long()]       # xbar of this layer comes from its own input coordinates
        dt_na, dt_ea = ctx.in_dtypes
        cast = lambda g, dt: None if g is None else g.to(dt)
        return (None, None, None, cast(g_na, dt_na), cast(g_ea, dt_ea), gh, gx, g_v, gZ, gS) + \
            tuple(views[n] for n in ctx.names)


def layer_call(named, flags: int, gravity, virtual_channels: int, graph: CsrGraph, h, x, v, Z, S, *, node_attr=None,
               attr_in=None, edge_attr_in=None):
    """(h', x', S', Z') of one layer from a dict of weight tensors keyed by the reference's state_dict suffixes
    (edge_mlp.0.weight, ...); S / S' in kernel layout [B,C,H].  Tensors must be contiguous fp32 CUDA.  node_attr: [N, Fa]
    contiguous fp32 CUDA tensor the kernels read, or None; node_mlp.0.weight then has Fa more columns.  attr_in /
    edge_attr_in: the tensors node_attr and graph.edge_attr were made from, to receive gradients (None: no gradient)."""
    names = tuple(named.keys())
    spec = (names, int(flags), gravity, int(virtual_channels))
    return _LayerFn.apply(spec, graph, node_attr, attr_in, edge_attr_in, _f32(h), _f32(x), _f32(v), _f32(Z), _f32(S),
                          *[named[n] for n in names])


def layer_forward(layer, node_feat, edge_index, coord, node_vel, virtual_coord, virtual_node_feat, data_batch,
                  edge_attr, node_attr=None, attr_in=None):
    """E_GCL_vel.forward: returns (node_feat, coord, virtual_node_feat, virtual_coord) (:223)."""
    L.deterministic("E_GCL_vel", L.NO_DET_LAYERS)
    _require_cuda(coord, "coord")
    B = int(virtual_coord.size(0))
    graph = CsrGraph(edge_index, data_batch, edge_attr, B)
    S = virtual_node_feat.permute(0, 2, 1).contiguous()        # [B,H,C] -> [B,C,H]
    flags = (L.F_ATTENTION if layer.attention else 0) | (L.F_NORMALIZE if layer.normalize else 0) | \
            (L.F_TANH if layer.tanh else 0) | (L.F_GRAVITY if layer.gravity is not None else 0) | \
            (L.F_COORDS_SUM if layer.coords_agg == 'sum' else 0)
    grav = None if layer.gravity is None else [float(t) for t in layer.gravity.detach().cpu().tolist()]
    named = dict(_layer_named(layer))
    h_new, x_new, S_new, Z_new = layer_call(named, flags, grav, layer.virtual_channels, graph, node_feat, coord, node_vel,
                                            virtual_coord, S.float(), node_attr=node_attr, attr_in=attr_in,
                                            edge_attr_in=edge_attr)
    return h_new, x_new, S_new.permute(0, 2, 1), Z_new
