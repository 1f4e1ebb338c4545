"""ROI occlusion on the fp64 oracle (oracle/gin_oracle.py): the reference the tests compare
GIN_InfoMaxReg.compute_roi_occlusion_batched with. It runs the oracle's eval-mode forward once on X and once per input
column d on X with column d set to 0, and restates nothing from the engine."""
import numpy as np
import torch

from oracle import gin_oracle
from graph_neural_mapping_b200.synth import SynthGraph


def roi_occlusion(state_dict, graphs, cls, cfg, cols=None, dtype=torch.float64):
    """Returns (out [B, D], f_x [B]): out[g, d] = (F_cls(X_g) - F_cls(X_g with column d set to 0)) / n_g for d in `cols`
    (default every column; the others are NaN), f_x the unoccluded scores. `cfg` is an oracle.gin_oracle.OracleConfig."""
    state = {k: (v.detach().clone().to(dtype) if v.is_floating_point() else v) for k, v in state_dict.items()}
    x = torch.cat([g.node_features for g in graphs], 0).to(dtype)

    def score(xx):
        return gin_oracle.forward(state, graphs, None, cfg, training=False, dtype=dtype, x_override=xx,
                                  with_dgi=False)["c_logit"][:, cls]

    with torch.no_grad():
        f_x = score(x)
        n = torch.tensor(np.diff(np.cumsum([0] + [len(g.g) for g in graphs])), dtype=dtype)
        out = torch.full((len(graphs), x.shape[1]), float("nan"), dtype=dtype)
        for d in (range(x.shape[1]) if cols is None else cols):
            xd = x.clone()
            xd[:, d] = 0
            out[:, d] = (f_x - score(xd)) / n
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
