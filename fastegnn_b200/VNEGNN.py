"""Host-side mirror of the reference VNEGNN sibling (models/VNEGNN.py of GLAD-RUC/FastEGNN; SURVEY.md 8 f3).

Same class names, constructor arguments, parameter creation order (hence the same initialisation under a seed) and
state_dict keys as the reference (:28-68 EGCL_A2A, :136-179 EGCL_A2V, :238-282 EGCL_V2A, :335-375 VNEGNN), so
utils/train.py:54-56 drives it unchanged.  Its three stages run on the SAME sm_100a phase kernels as FastEGNN: each stage
is one layer call (layer_fn.layer_call) whose weight table is assembled from the stage's parameters --

  A2A (:126-134)  real edges only: edge MLP, coordinate update by the MEAN of d_e phi_x(m_e), node update from
                  [h ; SUM_e m_e] (FEGNN_F_NODE_SUM).  Runs with one dummy virtual channel whose weights are zero.
  A2V (:210-225)  every real node to every virtual channel: u = phi([h ; S_c ; rho_c]) (FastEGNN's phi_ev without the M
                  columns: they are zero here), Z' = Z + mean_i D phi_X(u), S' = S + phi([S ; mean_i u]) (FastEGNN's phi_hv);
                  the real-side heads are zero and the graph has no edges.
  V2A (:318-328)  virtual to real: u2 from (h, S', Z'), x' = x + mean_c(-D phi(u2)) (FastEGNN's phi_xv head),
                  h' = h + phi([h ; mean_c u2]): FastEGNN's phi_h whose per-channel blocks all hold W / C.

The assembled tables are differentiable torch expressions of the parameters (cat / repeat_interleave with zeros), so the
hand-written backward of the phases reaches the real parameters through autograd.  Unused parts of a stage cost launches of
kernels that multiply by zero weights; a dedicated stage table would remove them (DESIGN.md).
"""
from __future__ import annotations

from typing import Dict

import torch
from torch import nn

from . import _lib as L
from .layer_fn import layer_call
from .ops import CsrGraph, _require_cuda

H = L.H


def _coord_mlp(hidden_nf, act_fn, use_tanh):
    last = nn.Linear(hidden_nf, 1, bias=False)                  # drawn BEFORE the HxH layer (:56-57)
    nn.init.xavier_uniform_(last.weight, gain=0.001)
    mods = [nn.Linear(hidden_nf, hidden_nf), act_fn, last]
    if use_tanh:
        mods.append(nn.Tanh())
    return nn.Sequential(*mods)


class _Stage(nn.Module):
    def __init__(self, node_feat_nf, node_feat_out_nf, node_attr_nf, edge_in, hidden_nf, virtual_channels, act_fn, residual,
                 attention, normalize, coords_agg, tanh):
        super().__init__()
        if hidden_nf != H or node_feat_nf != H or node_feat_out_nf != H:
            raise NotImplementedError(f"the sm_100a kernels are built for hidden_nf == {H}")
        if not isinstance(act_fn, nn.SiLU) or not residual or node_attr_nf != 0:
            raise NotImplementedError("act_fn=SiLU, residual=True, node_attr_nf=0 (what the reference mains use)")
        if attention:
            raise NotImplementedError("attention=True is not implemented for the VNEGNN stages")
        self.residual, self.attention, self.normalize, self.coords_agg, self.tanh = residual, attention, normalize, coords_agg, tanh
        self.hiddden_nf, self.node_feat_out_nf, self.epsilon = hidden_nf, node_feat_out_nf, 1e-8     # sic (:35)
        self.virtual_channels = virtual_channels
        self.edge_mlp = nn.Sequential(nn.Linear(edge_in, hidden_nf), act_fn, nn.Linear(hidden_nf, hidden_nf), act_fn)
        self.node_mlp = nn.Sequential(nn.Linear(2 * hidden_nf + node_attr_nf, hidden_nf), act_fn,
                                      nn.Linear(hidden_nf, node_feat_out_nf))
        self.coord_mlp = _coord_mlp(hidden_nf, act_fn, tanh)


class EGCL_A2A(_Stage):
    def __init__(self, node_feat_nf, node_feat_out_nf, node_attr_nf, edge_attr_nf, hidden_nf, virtual_channels,
                 act_fn=nn.SiLU(), residual=True, attention=False, normalize=False, coords_agg='mean', tanh=False):
        super().__init__(node_feat_nf, node_feat_out_nf, node_attr_nf, 2 * node_feat_nf + 1 + edge_attr_nf, hidden_nf,
                         virtual_channels, act_fn, residual, attention, normalize, coords_agg, tanh)


class EGCL_A2V(_Stage):
    def __init__(self, node_feat_nf, node_feat_out_nf, node_attr_nf, edge_attr_nf, hidden_nf, virtual_channels,
                 act_fn=nn.SiLU(), residual=True, attention=False, normalize=False, coords_agg='mean', tanh=False):
        super().__init__(node_feat_nf, node_feat_out_nf, 0, 2 * node_feat_nf + 1, hidden_nf, virtual_channels, act_fn,
                         residual, attention, normalize, coords_agg, tanh)


class EGCL_V2A(_Stage):
    def __init__(self, node_feat_nf, node_feat_out_nf, node_attr_nf, edge_attr_nf, hidden_nf, virtual_channels,
                 act_fn=nn.SiLU(), residual=True, attention=False, normalize=False, coords_agg='mean', tanh=False):
        super().__init__(node_feat_nf, node_feat_out_nf, node_attr_nf, 2 * node_feat_nf + 1, hidden_nf, virtual_channels,
                         act_fn, residual, attention, normalize, coords_agg, tanh)


def _zero_table(C: int, Fe: int, dev) -> Dict[str, torch.Tensor]:
    """A full FastEGNN layer table of zeros (a layer with these weights leaves h, x, S, Z unchanged)."""
    z = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float32)
    t = {"edge_mlp.0.weight": z(H, 2 * H + 1 + Fe), "edge_mlp.0.bias": z(H), "edge_mlp.2.weight": z(H, H), "edge_mlp.2.bias": z(H),
         "edge_mlp_virtual.0.weight": z(H, 2 * H + 1 + C), "edge_mlp_virtual.0.bias": z(H),
         "edge_mlp_virtual.2.weight": z(H, H), "edge_mlp_virtual.2.bias": z(H)}
    for head in ("coord_mlp_r", "coord_mlp_r_virtual", "coord_mlp_v_virtual"):
        t[f"{head}.0.weight"], t[f"{head}.0.bias"], t[f"{head}.2.weight"] = z(H, H), z(H), z(1, H)
    t.update({"coord_mlp_vel.0.weight": z(H, H), "coord_mlp_vel.0.bias": z(H), "coord_mlp_vel.2.weight": z(1, H),
              "coord_mlp_vel.2.bias": z(1),
              "node_mlp.0.weight": z(H, 2 * H + H * C), "node_mlp.0.bias": z(H), "node_mlp.2.weight": z(H, H), "node_mlp.2.bias": z(H),
              "node_mlp_virtual.0.weight": z(H, 2 * H), "node_mlp_virtual.0.bias": z(H),
              "node_mlp_virtual.2.weight": z(H, H), "node_mlp_virtual.2.bias": z(H)})
    return t


def _mlp(prefix: str, seq: nn.Sequential, first_weight=None) -> Dict[str, torch.Tensor]:
    out = {f"{prefix}.0.weight": seq[0].weight if first_weight is None else first_weight, f"{prefix}.0.bias": seq[0].bias,
           f"{prefix}.2.weight": seq[2].weight}
    if seq[2].bias is not None:
        out[f"{prefix}.2.bias"] = seq[2].bias
    return out


class VNEGNN(nn.Module):
    """Drop-in for the reference VNEGNN (:335-375): forward(node_feat, node_loc, edge_index, data_batch, virtual_node_loc,
    edge_attr=None, node_attr=None) -> (node_loc [N,3], virtual_node_loc [B,3,C])."""

    def __init__(self, node_feat_nf, node_attr_nf, edge_attr_nf, hidden_nf, virtual_channels, device='cpu', act_fn=nn.SiLU(),
                 n_layers=4, residual=True, attention=False, normalize=False, tanh=False):
        super().__init__()
        self.hidden_nf, self.device, self.n_layers, self.virtual_channels = hidden_nf, device, n_layers, virtual_channels
        assert virtual_channels > 0, f'Channels of virtual node must greater than 0 (got {virtual_channels})'
        if not 1 <= virtual_channels <= L.MAX_C:
            raise NotImplementedError(f"virtual_channels must be in [1, {L.MAX_C}]")
        self.virtual_node_feat = nn.Parameter(data=torch.randn(size=(1, hidden_nf, virtual_channels)), requires_grad=True)
        self.embedding_in = nn.Linear(node_feat_nf, hidden_nf)
        kw = dict(act_fn=act_fn, residual=residual, attention=attention, normalize=normalize, tanh=tanh)
        for i in range(n_layers):
            self.add_module(f'A2A_{i}', EGCL_A2A(hidden_nf, hidden_nf, node_attr_nf, edge_attr_nf, hidden_nf, virtual_channels, **kw))
            self.add_module(f'A2V_{i}', EGCL_A2V(hidden_nf, hidden_nf, node_attr_nf, edge_attr_nf, hidden_nf, virtual_channels, **kw))
            self.add_module(f'V2A_{i}', EGCL_V2A(hidden_nf, hidden_nf, node_attr_nf, edge_attr_nf, hidden_nf, virtual_channels, **kw))
        self._edge_attr_nf = edge_attr_nf
        self._flags = (L.F_NORMALIZE if normalize else 0) | (L.F_TANH if tanh else 0)
        self.to(self.device)

    def forward(self, node_feat, node_loc, edge_index, data_batch, virtual_node_loc, edge_attr=None, node_attr=None):
        L.deterministic("VNEGNN", L.NO_DET_LAYERS)
        _require_cuda(node_loc, "node_loc")
        dev = node_loc.device
        C, Fe = self.virtual_channels, self._edge_attr_nf
        B = int(virtual_node_loc.size(0))
        N = int(node_loc.size(0))
        if (edge_attr is None) != (Fe == 0):
            raise TypeError("edge_attr must be given exactly when edge_attr_nf > 0")
        graph = CsrGraph(edge_index, data_batch, edge_attr, B)                       # real edges: stage A2A
        no_edges = CsrGraph(edge_index[:, :0].contiguous(), data_batch, None, B)     # stages A2V / V2A: nodes only
        zero_v = torch.zeros(N, 3, device=dev)
        z1, zC, z0 = _zero_table(1, Fe, dev), _zero_table(C, 0, dev), None
        Zd, Sd = torch.zeros(B, 3, 1, device=dev), torch.zeros(B, 1, H, device=dev)  # dummy virtual channel of A2A
        S = self.virtual_node_feat[0].t().unsqueeze(0).expand(B, C, H).contiguous()  # [B,C,H] kernel layout (:364)
        Z = virtual_node_loc.float()
        h = torch.nn.functional.linear(node_feat.float(), self.embedding_in.weight, self.embedding_in.bias)   # :367
        x = node_loc.float()
        pad_m = torch.zeros(H, C, device=dev)                                        # the M columns FastEGNN's phi_ev has
        for i in range(self.n_layers):
            a2a, a2v, v2a = self._modules[f'A2A_{i}'], self._modules[f'A2V_{i}'], self._modules[f'V2A_{i}']
            # ---- A2A (:126-134)
            t = dict(z1)
            t.update(_mlp("edge_mlp", a2a.edge_mlp))
            t.update(_mlp("coord_mlp_r", a2a.coord_mlp))
            w0 = a2a.node_mlp[0].weight
            t.update(_mlp("node_mlp", a2a.node_mlp, torch.cat([w0, torch.zeros(H, H, device=dev)], dim=1).contiguous()))
            h, x, _, _ = layer_call(t, self._flags | L.F_NODE_SUM, None, 1, graph, h, x, zero_v, Zd, Sd)
            # ---- A2V (:210-225)
            t = dict(zC)
            t.update(_mlp("edge_mlp_virtual", a2v.edge_mlp, torch.cat([a2v.edge_mlp[0].weight, pad_m], dim=1).contiguous()))
            t.update(_mlp("coord_mlp_v_virtual", a2v.coord_mlp))
            t.update(_mlp("node_mlp_virtual", a2v.node_mlp))
            _, _, S, Z = layer_call(t, self._flags, None, C, no_edges, h, x, zero_v, Z, S)
            # ---- V2A (:318-328)
            t = dict(zC)
            t.update(_mlp("edge_mlp_virtual", v2a.edge_mlp, torch.cat([v2a.edge_mlp[0].weight, pad_m], dim=1).contiguous()))
            t.update(_mlp("coord_mlp_r_virtual", v2a.coord_mlp))
            w0 = v2a.node_mlp[0].weight                                              # [H, 2H]: [h ; mean_c u]
            w_exp = torch.cat([w0[:, :H], torch.zeros(H, H, device=dev), w0[:, H:].repeat_interleave(C, dim=1) / C], dim=1)
            t.update(_mlp("node_mlp", v2a.node_mlp, w_exp.contiguous()))
            h, x, _, _ = layer_call(t, self._flags, None, C, no_edges, h, x, zero_v, Z, S)
        return x, Z
