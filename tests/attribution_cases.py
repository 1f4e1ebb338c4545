"""Shared inputs of the attribution GPU tests (ROI saliency, integrated gradients, ROI occlusion): the model
configurations, seeded models and graphs, launch-count deltas and misaligned strided views."""
import torch

from graph_neural_mapping_b200 import ops, synth
from graph_neural_mapping_b200.models import GIN_InfoMaxReg
from graph_neural_mapping_b200.synth import SynthGraph

DEV = torch.device("cuda")

CONFIGS = {
    # name: (model kwargs, B, N, dense input width or None)
    "b1024_sum_tcgen05": (dict(), 1024, 400, None),
    "learn_eps": (dict(eps=True), 64, 400, None),
    "average_neighbour": (dict(neigh_pool="average"), 64, 400, None),
    "average_graph": (dict(graph_pool="average"), 64, 400, None),
    "max_neighbour": (dict(neigh_pool="max"), 8, 400, None),
    "mlp1": (dict(mlp=1), 64, 400, None),
    "mlp3_eps": (dict(mlp=3, eps=True), 64, 400, None),
    "dense_input_d400": (dict(), 32, 400, 400),
    "dense_input_d48_fused": (dict(eps=True), 32, 400, 48),
    "dense_input_max": (dict(neigh_pool="max"), 8, 200, 48),
    "n1000_f128": (dict(f=128), 8, 1000, None),
}


def make_model(d, f=64, layers=5, mlp=2, eps=False, graph_pool="sum", neigh_pool="sum", seed=0):
    torch.manual_seed(seed)
    m = GIN_InfoMaxReg(layers, mlp, d, f, 2, 0.0, eps, graph_pool, neigh_pool, DEV).to(DEV)
    with torch.no_grad():
        # eval BatchNorm with non-trivial running statistics and affine, so that the ReLU masks are mixed
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm1d):
                mod.running_mean.uniform_(-0.2, 0.2)
                mod.running_var.uniform_(0.5, 2.0)
                mod.weight.uniform_(0.5, 1.5)
                mod.bias.uniform_(-0.1, 0.2)
        m.eps.uniform_(-0.3, 0.3)
    return m


def graphs_of(b, n, seed=0, dense_dim=None, sparsity=30):
    gs = synth.make_graphs_bulk(b, n, sparsity, 128, seed0=seed, device=DEV)
    if dense_dim is not None:
        gen = torch.Generator().manual_seed(seed)
        gs = [SynthGraph(n, g.label, g.edge_mat, torch.rand(n, dense_dim, generator=gen)) for g in gs]
    return gs


def launches(fn):
    """(fn(), the launches per kernel family it made)."""
    before = ops.launch_counts()
    out = fn()
    torch.cuda.synchronize()
    return out, {k: v - before[k] for k, v in ops.launch_counts().items()}


def strided(m, w, pad, gen):
    """[m, w] view with leading dimension w + pad, starting one float into its buffer when pad > 0 (misaligned rows)."""
    off = 1 if pad else 0
    buf = torch.randn(m * (w + pad) + off, generator=gen).to(DEV)
    return buf[off:off + m * (w + pad)].view(m, w + pad)[:, :w]
