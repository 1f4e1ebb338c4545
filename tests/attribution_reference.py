"""Integrated gradients and ROI occlusion on the fp64 oracle (oracle/gin_oracle.py): the references the tests compare
GIN_InfoMaxReg.compute_integrated_gradients_batched and compute_roi_occlusion_batched with. Both evaluate the oracle's
eval-mode forward on modified node features and restate nothing from the engine."""
import numpy as np
import torch

from oracle import gin_oracle
from graph_neural_mapping_b200.synth import SynthGraph


def oracle_config(cfg):
    return gin_oracle.OracleConfig(cfg["num_layers"], cfg["num_mlp_layers"], cfg["input_dim"], cfg["hidden_dim"],
                                   cfg["output_dim"], cfg["final_dropout"], cfg["learn_eps"], cfg["graph_pooling_type"],
                                   cfg["neighbor_pooling_type"])


def score(state_dict, graphs, cls, cfg, dtype=torch.float64):
    """(f, x): x the graphs' node features in `dtype`, f(xx) the oracle's eval-mode class-`cls` scores [B] with node
    features xx in place of x. `cfg` is an oracle.gin_oracle.OracleConfig."""
    state = {k: (v.detach().clone().to(dtype) if v.is_floating_point() else v) for k, v in state_dict.items()}
    x = torch.cat([g.node_features for g in graphs], 0).to(dtype)

    def f(xx):
        return gin_oracle.forward(state, graphs, None, cfg, training=False, dtype=dtype, x_override=xx,
                                  with_dgi=False)["c_logit"][:, cls]
    return f, x


def integrated_gradients(state_dict, graphs, cls, cfg, steps, dtype=torch.float64):
    """Returns (out [B, D], delta [B], f_x [B], f_0 [B]): out[g] = (1/n_g) sum_{n in g} X[n] o (1/S) sum_s dF_cls/dX
    (alpha_s X)[n], alpha_s = (s + 1/2)/S; delta[g] = n_g sum_d out[g, d] - (F(X_g) - F(0)). Plain autograd at every
    path point x = alpha_s X (zero baseline, midpoint rule)."""
    f, x = score(state_dict, graphs, cls, cfg, dtype)
    grad_sum = torch.zeros_like(x)
    for s in range(steps):
        xa = (((s + 0.5) / steps) * x).requires_grad_(True)
        (g,) = torch.autograd.grad(f(xa).sum(), xa)          # graphs are independent in eval: per-graph gradients
        grad_sum += g
    attr = x * grad_sum / steps
    off = np.cumsum([0] + [len(g.g) for g in graphs])
    out = torch.stack([attr[off[i]:off[i + 1]].mean(0) for i in range(len(graphs))])
    with torch.no_grad():
        f_x, f_0 = f(x), f(torch.zeros_like(x))
    n = torch.tensor(np.diff(off), dtype=dtype)
    delta = n * out.sum(1) - (f_x - f_0)
    return out, delta, f_x, f_0


def roi_occlusion(state_dict, graphs, cls, cfg, cols=None, dtype=torch.float64):
    """Returns (out [B, D], f_x [B]): out[g, d] = (F_cls(X_g) - F_cls(X_g with column d set to 0)) / n_g for d in `cols`
    (default every column; the others are NaN), f_x the unoccluded scores. One forward on X and one per column."""
    f, x = score(state_dict, graphs, cls, cfg, dtype)
    with torch.no_grad():
        f_x = f(x)
        n = torch.tensor(np.diff(np.cumsum([0] + [len(g.g) for g in graphs])), dtype=dtype)
        out = torch.full((len(graphs), x.shape[1]), float("nan"), dtype=dtype)
        for d in (range(x.shape[1]) if cols is None else cols):
            xd = x.clone()
            xd[:, d] = 0
            out[:, d] = (f_x - f(xd)) / n
    return out, f_x


def with_neighbours(x):
    """Graph x with every node that has no neighbour joined to node 0 (node 1 for node 0 itself). The edge list keeps
    util.py:99-103's layout: the edges, then the same edges reversed."""
    em = x.edge_mat.cpu()
    half = em[:, :em.shape[1] // 2]
    lone = [i for i in range(len(x.g)) if not bool((em[0] == i).any())]
    add = torch.tensor([[i, 1 if i == 0 else 0] for i in lone], dtype=em.dtype).t().reshape(2, -1)
    first = torch.cat([half, add], 1)
    return SynthGraph(len(x.g), x.label, torch.cat([first, first.flip(0)], 1), x.node_features, with_neighbors=True)
