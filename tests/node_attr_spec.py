"""Specification of node attributes (node_attr_nf = Fa > 0) for the tests -- TEST INFRASTRUCTURE.

The reference's ``node_mlp.0`` is ``Linear(H + H + C*H + node_attr_nf, H)`` (models/FastEGNN.py:89-93); its input is
``[h ; mean_e m_e ; vec(u) ; a]``, the attribute columns LAST.  That order follows the constructor's width expression
and the EGNN convention; no golden vector of the unmodified reference covers node_attr_nf > 0, so it is UNPINNED
(DESIGN.md section 2), and this module is the specification the tests hold the kernels to.

Split by columns, with K = 2H + C*H,

    node_mlp.0([x ; a]) = W[:, :K] x + (b + W[:, K:] a),

so the attributes act as a per-node bias of the attribute-free Linear, and nothing else in the layer reads them.  The
model with attributes is stated here in exactly that form on top of ``oracle/fastegnn_oracle.py`` and
``oracle/staged.py``, which stay the attribute-free specification: every ``node_mlp.0.weight`` is replaced by its
leading K columns and ``node_mlp.0.bias`` by the [N, H] per-node bias ``b + a W[:, K:]^T`` (torch's linear broadcasts a
2-D bias over the rows).  Both are built with autograd from the original tensors, so the oracle's autograd gives the
gradient of the attribute columns; the staged backward adds it explicitly as dU1att = gUh^T a.
"""
from __future__ import annotations

from typing import Dict

import torch

from oracle import fastegnn_oracle as orc
from oracle import staged

T = torch.Tensor


def fold(params: Dict[str, T], node_attr: T) -> Dict[str, T]:
    """params with each node_mlp.0 written as the attribute-free Linear plus the per-node bias b + W[:, K:] a."""
    out = dict(params)
    Fa = node_attr.size(1)
    for key, W in params.items():
        if key == "node_mlp.0.weight" or key.endswith(".node_mlp.0.weight"):
            pre = key[:-len("weight")]
            K = W.size(1) - Fa
            out[key] = W[:, :K]
            out[pre + "bias"] = params[pre + "bias"] + node_attr @ W[:, K:].T
    return out


def oracle_forward(params, cfg: orc.OracleConfig, node_feat, node_loc, node_vel, edge_index, data_batch, loc_mean,
                   edge_attr, node_attr):
    """FastEGNN.forward (models/FastEGNN.py:265-276) with node attributes: (x [N,3], Z [B,3,C])."""
    return orc.fastegnn_forward(fold(params, node_attr), cfg, node_feat, node_loc, node_vel, edge_index, data_batch,
                                loc_mean, edge_attr)


def layer_forward(params, p: str, cfg: orc.OracleConfig, h, edge_index, x, v, Z, S, batch, edge_attr, node_attr):
    """One E_GCL_vel.forward (models/FastEGNN.py:192-223) with node attributes: (h', x', S', Z')."""
    return orc.layer_forward(fold(params, node_attr), p, cfg, h, edge_index, x, v, Z, S, batch, edge_attr)


def layer_weights(sd: Dict[str, T], node_attr: T, p: str, H: int, C: int, Fe: int, attention: bool, gravity: bool):
    """staged.LayerWeights of a layer with attributes: Uh = U1h h + (e1 + U1att a) through the per-node e1."""
    return staged.LayerWeights(fold(sd, node_attr), p, H, C, Fe, attention, gravity)


class StagedModel(staged.StagedModel):
    """staged.StagedModel with node attributes: the forward through the folded weights; the backward adds
    dU1att = gUh^T a (the attribute columns of node_mlp.0.weight) in every layer but the last, whose phi_h is dead."""

    def __init__(self, sd: Dict[str, T], node_attr: T, H, C, Fe, L, fl: staged.Flags):
        super().__init__(fold(sd, node_attr), H, C, Fe, L, fl)
        self.node_attr = node_attr

    def backward(self, gx_out, gZ_out):
        grads, gin = super().backward(gx_out, gZ_out)
        for l in range(self.L - 1):
            key = f"gcl_{l}.node_mlp.0.weight"
            gUh = self.bsaved[l]["b"]["gzh1"]
            grads[key] = torch.cat([grads[key], gUh.T @ self.node_attr], dim=1)
        return grads, gin
