"""Integrated gradients by plain autograd on the fp64 oracle (oracle/gin_oracle.py): the reference the tests compare
GIN_InfoMaxReg.compute_integrated_gradients_batched with. It evaluates the oracle's eval-mode forward at every path
point x = alpha_s X (zero baseline, midpoint rule) and restates nothing from the engine."""
import numpy as np
import torch

from oracle import gin_oracle


def oracle_config(cfg):
    return gin_oracle.OracleConfig(cfg["num_layers"], cfg["num_mlp_layers"], cfg["input_dim"], cfg["hidden_dim"],
                                   cfg["output_dim"], cfg["final_dropout"], cfg["learn_eps"], cfg["graph_pooling_type"],
                                   cfg["neighbor_pooling_type"])


def integrated_gradients(state_dict, graphs, cls, cfg, steps, dtype=torch.float64):
    """Returns (out [B, D], delta [B], f_x [B], f_0 [B]): out[g] = (1/n_g) sum_{n in g} X[n] o (1/S) sum_s dF_cls/dX
    (alpha_s X)[n], alpha_s = (s + 1/2)/S; delta[g] = n_g sum_d out[g, d] - (F(X_g) - F(0)). `cfg` is an
    oracle.gin_oracle.OracleConfig."""
    state = {k: (v.detach().clone().to(dtype) if v.is_floating_point() else v) for k, v in state_dict.items()}
    x = torch.cat([g.node_features for g in graphs], 0).to(dtype)

    def score(xx):
        return gin_oracle.forward(state, graphs, None, cfg, training=False, dtype=dtype, x_override=xx,
                                  with_dgi=False)["c_logit"][:, cls]

    grad_sum = torch.zeros_like(x)
    for s in range(steps):
        xa = (((s + 0.5) / steps) * x).requires_grad_(True)
        (g,) = torch.autograd.grad(score(xa).sum(), xa)      # graphs are independent in eval: per-graph gradients
        grad_sum += g
    attr = x * grad_sum / steps
    off = np.cumsum([0] + [len(g.g) for g in graphs])
    out = torch.stack([attr[off[i]:off[i + 1]].mean(0) for i in range(len(graphs))])
    with torch.no_grad():
        f_x, f_0 = score(x), score(torch.zeros_like(x))
    n = torch.tensor(np.diff(off), dtype=dtype)
    delta = n * out.sum(1) - (f_x - f_0)
    return out, delta, f_x, f_0
