"""Training through graphs built from positions: the torch composition a differentiable CsrGraph.from_radius stands for
(test infrastructure).  Each step's edge_attr is the edge length |x_row - x_col| of that step's positions in every
column, on a fixed edge list per step (the topology is piecewise constant); the velocity of the next step is the finite
difference of the positions."""
import torch


def lengths(x, ei, Fe):
    """edge_attr of a radius graph: torch's norm (its subgradient is 0 at a zero length) repeated over Fe columns."""
    return (x[ei[0]] - x[ei[1]]).norm(dim=1, keepdim=True).repeat(1, Fe)


def rollout(forward, x0, v0, lm0, edge_indices, Fe, dt):
    """len(edge_indices) steps of x_{t+1}, Z_{t+1} = forward(x_t, v_t, ei_t, lengths(x_t, ei_t), Z_t) with
    v_{t+1} = (x_{t+1} - x_t) / dt; returns the last (x, Z)."""
    x, v, Z = x0, v0, lm0
    for ei in edge_indices:
        x_new, Z = forward(x, v, ei, lengths(x, ei, Fe), Z)
        x, v = x_new, (x_new - x) / dt
    return x, Z
