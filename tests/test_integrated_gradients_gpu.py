"""Integrated gradients on the GPU: GIN_InfoMaxReg.compute_integrated_gradients_batched (path points as one virtual batch,
layer 0 once per real graph, gnm_ig_expand / gnm_ig_accumulate / gnm_ig_attribute) against the composed route of
existing code (compute_saliency_batched on alpha-scaled dense copies of the inputs), against plain autograd on the fp64
oracle, the completeness gap against class_logits, launch counts, reproducibility, and each kernel alone against
float64 torch."""
import ctypes

import numpy as np
import pytest
import torch

from attribution_cases import CONFIGS, DEV, graphs_of, launches, make_model, strided
from attribution_reference import integrated_gradients as ig_oracle, oracle_config
from helpers import Golden, assert_close, golden_names
from graph_neural_mapping_b200 import driver, lib, ops
from graph_neural_mapping_b200.models import GIN_InfoMaxReg
from graph_neural_mapping_b200.synth import SynthGraph

pytestmark = pytest.mark.gpu
TOL_GRAD = 3e-3
STEPS = 8


def assert_close_composed(a, b, what):
    """The composed route runs a different forward (alpha-scaled dense inputs through the dense aggregation and Linear)
    whose rounding can put a near-zero pre-activation on the other side of a ReLU kink than the one-hot call does; such
    a flip changes the gradient reaching every node of its graph at that path point, so it moves that graph's whole
    output row. So: every entry within 1e-3 of max-abs, and all graphs but 1 % of them (at least one) within 1e-4."""
    assert_close(a, b, 1e-3, what)
    a = np.nan_to_num(a.detach().cpu().numpy().astype(np.float64))
    b = np.nan_to_num(b.detach().cpu().numpy().astype(np.float64))
    far = (np.abs(a - b) > 1e-4 * max(float(np.abs(b).max()), 1e-30)).any(1)
    assert far.sum() <= max(1, len(far) // 100), "%s: %d of %d graphs differ by more than 1e-4 of max-abs" % (
        what, far.sum(), len(far))


def composed_route(model, graphs, classes, steps):
    """IG from existing code: compute_saliency_batched at x = alpha_s X (dense inputs), averaged over s, times X, averaged
    over each graph's nodes. [B, len(classes), D]."""
    x = torch.cat([g.node_features for g in graphs], 0).to(DEV)
    acc = [torch.zeros_like(x) for _ in classes]
    for s in range(steps):
        a = (s + 0.5) / steps
        scaled = [SynthGraph(len(g.g), g.label, g.edge_mat, a * g.node_features) for g in graphs]
        for k, cls in enumerate(classes):
            acc[k] += model.compute_saliency_batched(scaled, cls).detach()
    off = np.cumsum([0] + [len(g.g) for g in graphs])
    return torch.stack([torch.stack([(x * acc[k] / steps)[off[i]:off[i + 1]].mean(0) for k in range(len(classes))])
                        for i in range(len(graphs))])


ONEHOT_LINEAR = sorted(k for k, (kw, _, _, dense) in CONFIGS.items() if dense is None and kw.get("neigh_pool") != "max")


@pytest.mark.parametrize("name", ONEHOT_LINEAR)
def test_matches_composed_route(name):
    kw, b, n, _ = CONFIGS[name]
    model = make_model(n, **kw)
    graphs = graphs_of(b, n, seed=7)
    out = model.compute_integrated_gradients_batched(graphs, (0, 1), steps=STEPS)
    assert out.is_cuda and out.dtype == torch.float32 and tuple(out.shape) == (b, 2, n)
    ref = composed_route(model, graphs, (0, 1), STEPS)
    for k in (0, 1):
        assert_close_composed(out[:, k], ref[:, k], "%s class %d" % (name, k))


@pytest.mark.parametrize("name", [n for n in golden_names() if Golden(n).cfg["neighbor_pooling_type"] != "max"])
def test_against_fp64_oracle(name):
    g = Golden(name)
    c = g.cfg
    model = GIN_InfoMaxReg(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                           c["final_dropout"], c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"], DEV)
    sd = g.state_after_train()
    model.load_state_dict(sd)
    model = model.to(DEV)
    graphs = g.graphs()[:3]
    out, delta = model.compute_integrated_gradients_batched(graphs, (0, 1), steps=STEPS, return_delta=True)
    for k in (0, 1):
        ref, ref_delta, f_x, f_0 = ig_oracle(sd, graphs, k, oracle_config(c), STEPS)
        assert_close(out[:, k], ref, TOL_GRAD, "%s class %d" % (name, k))
        assert_close(delta[:, k], ref_delta, TOL_GRAD, "%s delta class %d" % (name, k),
                     floor=float((f_x.abs() + f_0.abs()).max()))


def test_delta_against_class_logits():
    n = 400
    model = make_model(n, seed=9)
    graphs = graphs_of(24, n, seed=5)
    out, delta = driver.integrated_gradients(model, graphs, classes=(0, 1), steps=16, batch=10, return_delta=True)
    zeros = [SynthGraph(n, g.label, g.edge_mat, torch.zeros(n, n)) for g in graphs]
    f_x = driver.class_logits(model, graphs).cpu().double().numpy()
    f_0 = driver.class_logits(model, zeros).cpu().double().numpy()
    expect = n * out.astype(np.float64).sum(2) - (f_x - f_0)
    assert_close(delta, expect, 1e-4, "delta", floor=float(np.abs(f_x).max() + np.abs(f_0).max()))


def test_isolated_nodes_average_learn_eps():
    """0/0 = NaN in the forward for a node without neighbours under average pooling (learn_eps: no self loops): NaN
    exactly where the composed route has NaN."""
    n = 400
    model = make_model(n, eps=True, neigh_pool="average", graph_pool="average", seed=5)
    graphs = []
    for i, g in enumerate(graphs_of(4, n, seed=21)):
        em = g.edge_mat
        if i % 2 == 0:
            cut = torch.tensor([0, 5, 17 + i])
            em = em[:, ~(torch.isin(em[0], cut) | torch.isin(em[1], cut))]
        graphs.append(SynthGraph(n, g.label, em.contiguous(), g.node_features))
    out = model.compute_integrated_gradients_batched(graphs, (0, 1), steps=4)
    ref = composed_route(model, graphs, (0, 1), 4)
    for k in (0, 1):
        assert_close_composed(out[:, k], ref[:, k], "class %d" % k)


def test_launch_counts_and_reproducibility():
    """At the benchmark shape: 50 points x 20 graphs x 400 nodes = one 1000-graph virtual batch per pass."""
    model = make_model(400, seed=1)
    graphs = graphs_of(40, 400, seed=3)
    model.compute_integrated_gradients_batched(graphs[:1], (0,), steps=2)
    a, ran = launches(lambda: model.compute_integrated_gradients_batched(graphs, (0, 1), steps=50))
    passes = chunks = 2
    assert ran["aggregate_tc"] > 0 and ran["linear_tc"] > 0, ran
    assert ran["linear_ffma"] == 0, ran                                       # no [M, 64] -> [M, 400] Linear
    assert ran["ig_expand"] == passes and ran["ig_accumulate"] == 2 * passes and ran["ig_attribute"] == 2 * chunks, ran
    assert not ops.aggregate_tc_status()
    b = model.compute_integrated_gradients_batched(graphs, (0, 1), steps=50)
    assert torch.equal(a, b)


def test_parameter_gradients_untouched():
    model = make_model(400, seed=2)
    graphs = graphs_of(8, 400, seed=4)
    model.compute_saliency([graphs[0]], 1)
    model.eps.grad = None
    before = {k: (None if p.grad is None else p.grad.clone()) for k, p in model.named_parameters()}
    model.train()
    model.compute_integrated_gradients_batched(graphs, (0, 1), steps=4)
    assert not model.training
    for k, p in model.named_parameters():
        assert (p.grad is None) == (before[k] is None) and (p.grad is None or torch.equal(p.grad, before[k])), k


# ---- the kernels alone ----------------------------------------------------------------------------------------------

COUNTS = [5, 0, 400, 1, 0, 37, 129, 2]


def _offsets():
    counts = torch.tensor(COUNTS)
    return counts, torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)]).to(torch.int32).to(DEV)


@pytest.mark.parametrize("width", [1, 3, 64, 128])
@pytest.mark.parametrize("pad", [0, 3])
def test_expand_and_accumulate_against_torch(width, pad):
    gen = torch.Generator().manual_seed(width * 10 + pad)
    counts, node_off = _offsets()
    m, points = int(counts.sum()), 5
    p = strided(m, width, pad, gen)
    bias = torch.randn(width, generator=gen).to(DEV)
    alpha = torch.rand(points, generator=gen).to(DEV)
    no = node_off.long().tolist()
    z = strided(points * m, width, pad, gen)
    ops.ig_expand(p, bias, alpha, node_off, points, z)
    ref = torch.cat([alpha[s].double() * p[no[g]:no[g + 1]].double() + bias.double()
                     for g in range(len(COUNTS)) for s in range(points)])
    assert_close(z, ref.cpu(), 1e-6, "expand")
    dy = strided(points * m, width, pad, gen)
    coef = torch.randn(3, width, generator=gen).to(DEV)
    out = strided(m, width, pad, gen)
    ops.ig_accumulate(dy, coef, node_off, points, 0.25, out, False)
    ref = torch.cat([0.25 * coef[0].double() * dy[points * no[g]:points * no[g + 1]].double().view(points, COUNTS[g], width).sum(0)
                     for g in range(len(COUNTS))])
    assert_close(out, ref.cpu(), 1e-5, "accumulate")
    ops.ig_accumulate(dy, None, node_off, points, 0.5, out, True)
    ref = ref + torch.cat([0.5 * dy[points * no[g]:points * no[g + 1]].double().view(points, COUNTS[g], width).sum(0)
                           for g in range(len(COUNTS))])
    assert_close(out, ref.cpu(), 1e-5, "accumulate on top")


@pytest.mark.parametrize("width", [1, 3, 64, 128])
@pytest.mark.parametrize("pad", [0, 3])
def test_attribute_against_torch(width, pad):
    gen = torch.Generator().manual_seed(width * 10 + pad + 1)
    counts, node_off = _offsets()
    m, d = int(counts.sum()), 450
    t = strided(m, width, pad, gen)
    table = strided(d, width, pad, gen)
    tags = torch.randint(0, d, (m,), generator=gen)
    tags[400:410] = 3                                          # duplicate tags inside the 400-node graph
    tags = tags.to(torch.int32).to(DEV)
    out = torch.full((len(COUNTS), d + 2), 7.0, device=DEV)[:, :d]
    ops.ig_attribute(t, table, tags, node_off, out)
    a = (t.double() * table.double()[tags.long()]).sum(1)
    no = node_off.long().tolist()
    ref = torch.zeros(len(COUNTS), d, dtype=torch.float64, device=DEV)
    for g in range(len(COUNTS)):
        ref[g].index_add_(0, tags[no[g]:no[g + 1]].long(), a[no[g]:no[g + 1]])
        ref[g] /= max(COUNTS[g], 1)
    assert_close(out, ref.cpu(), 1e-5, "attribute")
    assert bool((out[(counts == 0).to(DEV)] == 0).all()), "empty graphs must give zeros"
    t2 = t.clone()
    t2[no[5] + 3, 0] = float("inf")
    ops.ig_attribute(t2, table, tags, node_off, out)
    assert bool(torch.isnan(out[5]).all()) and not bool(torch.isnan(out[torch.arange(8) != 5]).any())


def test_kernel_argument_checks():
    l = lib.load()
    p = ctypes.c_void_p
    x = torch.zeros(16, 4, device=DEV)
    node_off = torch.tensor([0, 4, 8], dtype=torch.int32, device=DEV)
    st = p(torch.cuda.current_stream().cuda_stream)
    before = ops.launch_counts()
    assert l.gnm_ig_expand(p(x.data_ptr()), 4, None, p(x.data_ptr()), p(node_off.data_ptr()), 2, 8, -1, 4,
                           p(x.data_ptr()), 4, st) == -1
    assert l.gnm_ig_accumulate(p(x.data_ptr()), 4, None, p(node_off.data_ptr()), 2, 8, 2, 0, 1.0, 0, p(x.data_ptr()), 4,
                               st) == 0
    assert l.gnm_ig_attribute(p(x.data_ptr()), 4, p(x.data_ptr()), 4, 0, p(node_off.data_ptr()), p(node_off.data_ptr()), 2,
                              4, p(x.data_ptr()), 4, st) == 0
    assert ops.launch_counts() == before, "an empty or rejected problem must launch nothing"
