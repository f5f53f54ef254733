"""Host-side mirror of the reference module API (models/FastEGNN.py of GLAD-RUC/FastEGNN).

Same class names, constructor arguments, forward signatures, parameter creation order
(hence the same random initialisation under a seed) and state_dict keys as the
reference (:6-99, :226-276), so `from models.FastEGNN import FastEGNN` keeps working for
main_nbody.py / main_protein.py / main_simulation.py, utils/train.py and
equivariant_test.py.  All arithmetic runs in libfegnn.so (hand-written sm_100a kernels,
explicit backward); there is no eager / CPU fallback -- non-CUDA tensors raise.

Differences a caller can observe
  * hidden_nf must be 64, act_fn must be SiLU, residual must be True (what all three mains use) and node_attr_nf
    at most 16; anything else raises NotImplementedError.
  * node_attr (node_attr_nf > 0) enters node_mlp.0 as its LAST node_attr_nf input columns, [h ; mean m ; vec(u) ; a]
    (:89-93,:159).  That order is restated from the constructor's width expression and is unpinned: no golden vector
    of the unmodified reference covers node_attr_nf > 0.
  * node_vel, node_attr and edge_attr receive gradients as in the reference, computed only when they require grad
    (fegnn_model_backward_inputs).  Exceptions: FastRF's node_vel (none), and the edge_attr a prebuilt CsrGraph carries
    (data of the graph: pass graph.edge_index() and a tensor to differentiate it).
  * the number of graphs is taken from loc_mean.size(0) instead of data_batch[-1].item()
    (:267), which removes a device synchronisation; the two agree for valid batches.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional

import torch
from torch import nn

from . import _lib as L
from .ops import (CsrGraph, SavedBlock, _on, _require_cuda, _stream, layer_ptrs, make_dims, node_attr_arg,
                  segment_reduce)

lib = L.lib


def _coord_head(hidden_nf: int, act_fn: nn.Module, use_tanh: bool) -> nn.Sequential:
    # RNG order matters: the 1-wide output layer is drawn before the HxH layer (:56-60)
    out = nn.Linear(hidden_nf, 1, bias=False)
    nn.init.xavier_uniform_(out.weight, gain=0.001)
    mods = [nn.Linear(hidden_nf, hidden_nf), act_fn, out]
    if use_tanh:
        mods.append(nn.Tanh())
    return nn.Sequential(*mods)


def _flags(attention: bool, normalize: bool, tanh: bool, gravity) -> int:
    return ((L.F_ATTENTION if attention else 0) | (L.F_NORMALIZE if normalize else 0) | (L.F_TANH if tanh else 0) |
            (L.F_GRAVITY if gravity is not None else 0))


def _gravity_list(gravity):
    if gravity is None:
        return None
    if isinstance(gravity, torch.Tensor):
        return [float(v) for v in gravity.detach().cpu().tolist()]
    return [float(v) for v in gravity]


class E_GCL_vel(nn.Module):
    """One FastEGNN layer; parameter container + layer-level entry point (:6-223)."""

    def __init__(self, node_feat_nf, node_feat_out_nf, node_attr_nf, edge_attr_nf, hidden_nf, virtual_channels,
                 act_fn=nn.SiLU(), residual=True, attention=False, normalize=False, coords_agg='mean', tanh=False,
                 gravity=None):
        super().__init__()
        if hidden_nf != L.H or node_feat_nf != L.H or node_feat_out_nf != L.H:
            raise NotImplementedError(f"the sm_100a kernels are built for hidden_nf == {L.H} "
                                      f"(got in={node_feat_nf}, out={node_feat_out_nf}, hidden={hidden_nf})")
        if not isinstance(act_fn, nn.SiLU):
            raise NotImplementedError("only act_fn=nn.SiLU() is implemented (the reference default, used by all mains)")
        if not residual:
            raise NotImplementedError("residual=False is not implemented (all reference mains use residual=True)")
        if not 0 <= node_attr_nf <= L.MAX_FA:
            raise NotImplementedError(f"node_attr_nf must be in [0, {L.MAX_FA}]")
        if not 1 <= virtual_channels <= L.MAX_C:
            raise NotImplementedError(f"virtual_channels must be in [1, {L.MAX_C}]")
        if not 0 <= edge_attr_nf <= L.MAX_FE:
            raise NotImplementedError(f"edge_attr_nf must be in [0, {L.MAX_FE}]")
        self.residual, self.attention, self.normalize, self.coords_agg, self.tanh = \
            residual, attention, normalize, coords_agg, tanh
        self.hiddden_nf = hidden_nf            # sic -- attribute name of the reference (:18)
        self.node_feat_out_nf = node_feat_out_nf
        self.epsilon = 1e-8
        self.virtual_channels = virtual_channels
        self.edge_attr_nf = edge_attr_nf
        self.node_attr_nf = node_attr_nf
        H, Cc = hidden_nf, virtual_channels
        self.edge_mlp = nn.Sequential(nn.Linear(2 * H + 1 + edge_attr_nf, H), act_fn, nn.Linear(H, H), act_fn)
        self.edge_mlp_virtual = nn.Sequential(nn.Linear(2 * H + 1 + Cc, H), act_fn, nn.Linear(H, H), act_fn)
        if attention:
            self.att_mlp = nn.Sequential(nn.Linear(H, 1), nn.Sigmoid())
            self.att_mlp_virtual = nn.Sequential(nn.Linear(H, 1), nn.Sigmoid())
        self.coord_mlp_r = _coord_head(H, act_fn, tanh)
        self.coord_mlp_r_virtual = _coord_head(H, act_fn, tanh)
        self.coord_mlp_v_virtual = _coord_head(H, act_fn, tanh)
        self.coord_mlp_vel = nn.Sequential(nn.Linear(H, H), act_fn, nn.Linear(H, 1))
        self.gravity = gravity
        if gravity is not None:
            self.gravity_mlp = nn.Sequential(nn.Linear(H, H), act_fn, nn.Linear(H, 1))
        self.node_mlp = nn.Sequential(nn.Linear(H + H + Cc * H + node_attr_nf, H), act_fn, nn.Linear(H, node_feat_out_nf))
        self.node_mlp_virtual = nn.Sequential(nn.Linear(2 * H, H), act_fn, nn.Linear(H, node_feat_out_nf))

    def forward(self, node_feat, edge_index, coord, node_vel, virtual_coord, virtual_node_feat, data_batch,
                edge_attr=None, node_attr=None):
        """(h, x, S, Z) of one layer, S in the reference's [B,H,C] layout (:192-223)."""
        if self.coords_agg not in ('sum', 'mean'):
            raise Exception('Wrong coords_agg parameter')      # raised at call time with the reference's text (:131)
        attr_in = node_attr
        node_attr = node_attr_arg(node_attr, self.node_attr_nf, coord.size(0))
        from .layer_fn import layer_forward     # phase-by-phase driver (also used by the partitioned path)
        return layer_forward(self, node_feat, edge_index, coord, node_vel, virtual_coord, virtual_node_feat,
                             data_batch, edge_attr, node_attr, attr_in)


class _StackFn(torch.autograd.Function):
    """FastEGNN.forward / backward as two C calls (fegnn_model_forward / fegnn_model_backward_inputs).

    node_attr is the contiguous fp32 copy the kernels read; attr_in / edge_attr_in are the caller's tensors (or None), which
    are inputs here only so that autograd can hand them their gradients.  The kernels read edge_attr from the graph.
    With mod.recompute the flag word carries FEGNN_F_RECOMPUTE: the workspace holds the states and two saved blocks, and
    the backward (which reads the flag from ctx.dims, not from the module) rebuilds each layer's block.  A recompute
    backward leaves the two blocks holding other layers than the forward did, so a further backward over the same graph
    (retain_graph=True) passes FEGNN_F_REBUILD_ALL and rebuilds every layer."""

    @staticmethod
    def forward(ctx, mod: "FastEGNN", graph: CsrGraph, node_attr, attr_in, edge_attr_in, node_feat, x0, v, loc_mean,
                *params):
        dev = x0.device
        N, B, Cc, Lyr = graph.N, graph.B, mod.virtual_channels, mod.n_layers
        recompute = bool(mod.recompute)
        flags = mod._flag_word | (L.F_RECOMPUTE if recompute else 0)
        dims = make_dims(N, N, graph.E, B, Cc, graph.Fe, flags, mod._gravity, Fa=mod._node_attr_nf, node_attr=node_attr)
        pd = C.byref(dims)
        table, names = mod._param_table()
        ws_floats = int(lib.fegnn_model_workspace_floats(pd, Lyr))
        ws = torch.empty(ws_floats, device=dev, dtype=torch.float32)
        x_out = torch.empty(N, 3, device=dev, dtype=torch.float32)
        Z_out = torch.empty(B, 3, Cc, device=dev, dtype=torch.float32)
        Fin = node_feat.size(1)
        with _on(dev):
            L.check(lib.fegnn_model_forward(pd, Lyr, Fin, C.byref(graph.c), table, L.ptr(mod.embedding_in.weight),
                                            L.ptr(mod.embedding_in.bias), L.ptr(mod.virtual_node_feat), L.ptr(node_feat),
                                            L.ptr(x0), L.ptr(v), L.ptr(loc_mean), L.ptr(x_out), L.ptr(Z_out), L.ptr(ws),
                                            ws_floats, _stream(dev)), "fegnn_model_forward")
        ctx.mod, ctx.graph, ctx.dims, ctx.ws, ctx.Fin = mod, graph, dims, ws, Fin
        ctx.recompute = recompute                               # the backward follows this step's forward
        ctx.blocks_consumed = False                             # recompute: set by the first backward (see above)
        ctx.save_for_backward(node_feat, v, node_attr)          # node_attr: dims points at it until the backward
        ctx.names = names
        ctx.need_nf = node_feat.requires_grad
        ctx.in_dtypes = (None if attr_in is None else attr_in.dtype, None if edge_attr_in is None else edge_attr_in.dtype,
                         v.dtype)
        ctx.mark_non_differentiable()
        return x_out, Z_out

    @staticmethod
    def backward(ctx, gx, gZ):
        mod, graph, dims = ctx.mod, ctx.graph, ctx.dims
        L.deterministic(type(mod).__name__ + " backward", L.NO_DET_LAYERS)
        node_feat, v, _ = ctx.saved_tensors
        dev = v.device
        N, B, Cc, Lyr = graph.N, graph.B, mod.virtual_channels, mod.n_layers
        if ctx.recompute and ctx.blocks_consumed:
            dims = type(dims).from_buffer_copy(dims)
            dims.flags |= L.F_REBUILD_ALL
        pd = C.byref(dims)
        gx = torch.zeros(N, 3, device=dev) if gx is None else gx.contiguous().float()
        gZ = torch.zeros(B, 3, Cc, device=dev) if gZ is None else gZ.contiguous().float()
        table, names = mod._param_table()
        flat, views, gtable = mod._grad_table(dev)
        scr_floats = int(lib.fegnn_model_backward_scratch_floats(pd))
        scratch = torch.empty(scr_floats, device=dev, dtype=torch.float32)
        g_x0 = torch.empty(N, 3, device=dev, dtype=torch.float32)
        g_lm = torch.empty(B, 3, Cc, device=dev, dtype=torch.float32)
        g_nf = torch.empty_like(node_feat) if ctx.need_nf else None
        # the input gradients exactly as requested; FastRF's velocity enters through |v| and has none (not implemented)
        need = ctx.needs_input_grad
        f32 = dict(device=dev, dtype=torch.float32)
        g_na = torch.empty(N, dims.Fa, **f32) if need[3] else None
        g_ea = (torch.empty if graph.Fe else torch.zeros)(graph.E, graph.Fe, **f32) if need[4] else None
        g_v = torch.empty(N, 3, **f32) if need[7] and not (mod._flag_word & L.F_RF) else None
        ig = L.InputGrads(L.ptr(g_v), L.ptr(g_na), L.ptr(g_ea) if graph.Fe else None, L.ptr(graph.perm))
        with _on(dev):
            L.check(lib.fegnn_model_backward_inputs(pd, Lyr, ctx.Fin, C.byref(graph.c), table, gtable,
                                                    L.ptr(mod.embedding_in.weight), L.ptr(views["embedding_in.weight"]),
                                                    L.ptr(views["embedding_in.bias"]), L.ptr(views["virtual_node_feat"]),
                                                    L.ptr(node_feat), L.ptr(v), L.ptr(gx), L.ptr(gZ), L.ptr(g_x0),
                                                    L.ptr(g_lm), L.ptr(g_nf), L.ptr(ctx.ws), L.ptr(scratch), scr_floats,
                                                    C.byref(ig), _stream(dev)), "fegnn_model_backward_inputs")
        ctx.blocks_consumed = ctx.recompute
        dead = mod._dead_names
        grads = tuple(None if n in dead else views[n] for n in names)
        dt_na, dt_ea, dt_v = ctx.in_dtypes
        cast = lambda g, dt: None if g is None else g.to(dt)
        return (None, None, None, cast(g_na, dt_na), cast(g_ea, dt_ea), g_nf, g_x0, cast(g_v, dt_v), g_lm) + grads


def _stack_inference(mod: "FastEGNN", graph: CsrGraph, node_attr, node_feat, x0, v, loc_mean):
    """FastEGNN.forward without autograd: fegnn_model_forward_inference (two ping-pong states + one shared block of
    per-layer intermediates -- a ring of four blocks up to 65 536 nodes; nothing is kept for a backward)."""
    dev = x0.device
    N, B, Cc, Lyr = graph.N, graph.B, mod.virtual_channels, mod.n_layers
    dims = make_dims(N, N, graph.E, B, Cc, graph.Fe, mod._flag_word, mod._gravity, Fa=mod._node_attr_nf,
                     node_attr=node_attr)
    pd = C.byref(dims)
    table, _ = mod._param_table()
    # + the scratch of the deterministic kernels, behind it (0 with the mode off)
    ws_floats = int(lib.fegnn_model_inference_workspace_floats(pd)) + int(lib.fegnn_model_inference_det_workspace_floats(pd))
    ws = torch.empty(ws_floats, device=dev, dtype=torch.float32)
    x_out = torch.empty(N, 3, device=dev, dtype=torch.float32)
    Z_out = torch.empty(B, 3, Cc, device=dev, dtype=torch.float32)
    with _on(dev):
        L.check(lib.fegnn_model_forward_inference(pd, Lyr, node_feat.size(1), C.byref(graph.c), table,
                                                  L.ptr(mod.embedding_in.weight), L.ptr(mod.embedding_in.bias),
                                                  L.ptr(mod.virtual_node_feat), L.ptr(node_feat), L.ptr(x0), L.ptr(v),
                                                  L.ptr(loc_mean), L.ptr(x_out), L.ptr(Z_out), L.ptr(ws), ws_floats,
                                                  _stream(dev)), "fegnn_model_forward_inference")
    return x_out, Z_out


class FastEGNN(nn.Module):
    """Drop-in for the reference FastEGNN (:226-276).

    eval_keeps_graph (attribute, default False): the reference's evaluation epochs (utils/train.py:24-27,191-192) run the
    model under model.eval() WITHOUT torch.no_grad(), building an autograd graph nobody uses.  Here a forward in eval mode
    -- or under torch.no_grad() -- takes the forward-only stack (fegnn_model_forward_inference): same outputs, no saved
    activations, outputs without grad_fn.  Set eval_keeps_graph = True to get the training forward in eval mode.

    recompute (attribute, default False): activation checkpointing for the training stack.  The forward keeps only the
    n_layers + 1 layer states and the backward rebuilds each layer's intermediates just before that layer's backward, so a
    step holds two saved blocks instead of n_layers (about 1.5 KB + 256 B * virtual_channels per node each) for about one
    more forward per step (DESIGN 3.8).  Same results up to float summation order.  A step's backward follows the setting
    of its forward.  The eval() / no_grad forward-only stack is unaffected."""
    eval_keeps_graph = False
    recompute = False
    _node_attr_nf = 0          # subclasses without node attributes (FastRF) inherit forward and the stack functions

    def __init__(self, node_feat_nf, node_attr_nf, edge_attr_nf, hidden_nf, virtual_channels, device='cpu',
                 act_fn=nn.SiLU(), n_layers=4, residual=True, attention=False, normalize=False, tanh=False,
                 gravity=None):
        super().__init__()
        self.hidden_nf = hidden_nf
        self.device = device
        self.n_layers = n_layers
        self.virtual_channels = virtual_channels
        assert virtual_channels > 0, f'Channels of virtual node must greater than 0 (got {virtual_channels})'
        if not 1 <= n_layers <= 32:
            raise NotImplementedError("n_layers must be in [1, 32]")
        if not 1 <= node_feat_nf <= 16:
            raise NotImplementedError("node_feat_nf must be in [1, 16]")
        self.virtual_node_feat = nn.Parameter(data=torch.randn(size=(1, hidden_nf, virtual_channels)),
                                              requires_grad=True)
        self.embedding_in = nn.Linear(node_feat_nf, hidden_nf)
        self._gravity = _gravity_list(gravity)
        if gravity is not None:
            gravity = torch.tensor(gravity, device=device)       # same attribute type as :258-259
        for i in range(n_layers):
            self.add_module("gcl_%d" % i, E_GCL_vel(hidden_nf, hidden_nf, node_attr_nf, edge_attr_nf, hidden_nf,
                                                    virtual_channels=virtual_channels, act_fn=act_fn,
                                                    residual=residual, attention=attention, normalize=normalize,
                                                    tanh=tanh, gravity=gravity))
        self._flag_word = _flags(attention, normalize, tanh, gravity)
        self._edge_attr_nf = edge_attr_nf
        self._node_attr_nf = node_attr_nf
        self._cache = None
        last = "gcl_%d" % (n_layers - 1)
        # the final h and S are discarded (:276): these tensors receive no gradient in the reference
        self._dead_names = frozenset(f"{last}.{m}.{i}.{k}" for m in ("node_mlp", "node_mlp_virtual")
                                     for i in (0, 2) for k in ("weight", "bias"))
        self.to(self.device)

    # -- pointer tables -------------------------------------------------------------------
    def _apply(self, fn, *a, **k):
        self._cache = None          # .to() / .cuda() / .float() re-allocate parameter storage
        return super()._apply(fn, *a, **k)

    def _signature_tensors(self):
        return (self.virtual_node_feat, self.embedding_in.weight,
                getattr(self, "gcl_%d" % (self.n_layers - 1)).node_mlp_virtual[2].bias)

    def _param_table(self):
        """(fegnn_layer_params[L], ordered parameter names).  Cached; storage addresses are
        stable under optimizer steps and load_state_dict (both write in place)."""
        named = dict(self.named_parameters())
        sig = tuple(p.data_ptr() for p in self._signature_tensors())
        if self._cache is None or self._cache[0] != sig:
            for n, p in named.items():
                if not p.is_cuda or p.dtype != torch.float32:
                    raise L.FegnnError(f"parameter {n} is {p.dtype} on {p.device}: the model must be fp32 on a CUDA "
                                       "device (construct it with device='cuda:0'); there is no CPU path")
            table = (L.LayerPtrs * self.n_layers)()
            for l in range(self.n_layers):
                table[l] = layer_ptrs(named, "gcl_%d" % l)
            names = list(named.keys())
            sizes = [named[n].numel() for n in names]
            self._cache = (sig, table, names, sizes)
        return self._cache[1], self._cache[2]

    def _grad_table(self, device):
        """One zero-filled flat buffer with a view per parameter + fegnn_layer_grads[L] into it."""
        _, _, names, sizes = self._cache
        named = dict(self.named_parameters())
        offs, tot = [], 0
        for s in sizes:
            offs.append(tot)
            tot += (s + 3) & ~3           # keep every view 16-byte aligned
        flat = torch.zeros(tot, device=device, dtype=torch.float32)
        views = {n: flat[o:o + s].view_as(named[n]) for n, o, s in zip(names, offs, sizes)}
        gtable = (L.LayerPtrs * self.n_layers)()
        for l in range(self.n_layers):
            gtable[l] = layer_ptrs({k: v for k, v in views.items() if k not in self._dead_names}, "gcl_%d" % l)
        return flat, views, gtable

    # -- forward --------------------------------------------------------------------------
    def _inference_route(self):
        """True when forward takes the forward-only stack (no autograd graph)."""
        return not torch.is_grad_enabled() or (not self.training and not self.eval_keeps_graph)

    def forward(self, node_feat, node_loc, node_vel, edge_index, data_batch, loc_mean, edge_attr=None, node_attr=None):
        # the forward-only stack has deterministic forms of its kernels; the training forward and its backward have none
        L.deterministic(type(self).__name__, None if self._inference_route() else L.NO_DET_LAYERS)
        attr_in = node_attr
        node_attr = node_attr_arg(node_attr, self._node_attr_nf, node_loc.size(0))
        _require_cuda(node_loc, "node_loc")
        if isinstance(edge_index, CsrGraph):
            # a graph already in kernel layout (CsrGraph.from_radius, or a CsrGraph reused across steps of a static
            # batch): no per-forward sort.  Its edge_attr is used; the edge_attr argument must be None.
            graph = edge_index
            if edge_attr is not None:
                raise TypeError("edge_attr must be None when edge_index is a prebuilt CsrGraph (it carries its own)")
            if graph.Fe != self._edge_attr_nf or graph.N != node_loc.size(0) or graph.B != loc_mean.size(0):
                raise RuntimeError(f"prebuilt graph (N={graph.N}, B={graph.B}, Fe={graph.Fe}) does not match the inputs "
                                   f"(N={node_loc.size(0)}, B={loc_mean.size(0)}, edge_attr_nf={self._edge_attr_nf})")
            # node_attr still gets its gradient; the graph's edge_attr is data of the graph (no autograd input here)
            return self._run_stack(graph, node_attr, attr_in, None, node_feat, node_loc, node_vel, loc_mean)
        if edge_attr is None:
            if self._edge_attr_nf != 0:
                raise TypeError("edge_attr is required when edge_attr_nf > 0 (the reference's torch.cat fails on None, "
                                "models/FastEGNN.py:103)")
        elif edge_attr.size(1) != self._edge_attr_nf:
            raise RuntimeError(f"edge_attr has {edge_attr.size(1)} columns, model was built with edge_attr_nf="
                               f"{self._edge_attr_nf}")
        B = int(loc_mean.size(0))
        graph = CsrGraph(edge_index, data_batch, edge_attr, B, overlap=True)      # the sort runs under the first node phase
        return self._run_stack(graph, node_attr, attr_in, edge_attr, node_feat, node_loc, node_vel, loc_mean)

    def _run_stack(self, graph, node_attr, attr_in, edge_attr_in, node_feat, node_loc, node_vel, loc_mean):
        args = (node_feat.contiguous().float(), node_loc.contiguous().float(), node_vel.contiguous().float(),
                loc_mean.contiguous().float())
        try:
            if self._inference_route():
                return _stack_inference(self, graph, node_attr, *[a.detach() for a in args])
            params = [p for _, p in self.named_parameters()]
            return _StackFn.apply(self, graph, node_attr, attr_in, edge_attr_in, *args, *params)
        finally:
            # the C call has joined the side stream of CsrGraph(overlap=True): later users of the graph (backward) need no wait
            if getattr(graph, "_ready", None) is not None:
                graph._ready = None
                graph.c.ready_event = None


def unsorted_segment_sum(data, segment_ids, num_segments):
    """models/FastEGNN.py:279-284: rows of `data` [E,K] summed per segment -> [num_segments,K].  Module-level helper of
    the reference file (the layer's own sums run inside the fused edge kernel); here fegnn_segment_sum: one warp per
    row, red.global.add.  CUDA fp32 only, like everything in this package."""
    return segment_reduce(data, segment_ids, num_segments, mean=False)


def unsorted_segment_mean(data, segment_ids, num_segments):
    """models/FastEGNN.py:287-294: segment sums divided by the per-segment count clamped to >= 1."""
    return segment_reduce(data, segment_ids, num_segments, mean=True)
