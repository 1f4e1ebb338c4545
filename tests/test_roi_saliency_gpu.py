"""ROI saliency on the GPU: GIN_InfoMaxReg.compute_roi_saliency_batched (one eval forward, one backward per class, layer 0
reduced per graph by gnm_segment_weighted_colsum) against the node average of the full saliency maps of the same code
path, against the reference's maps in the golden fixtures and the fp64 oracle, and the kernel alone against torch."""
import ctypes

import numpy as np
import pytest
import torch

from attribution_cases import CONFIGS, DEV, graphs_of, launches, make_model, strided
from attribution_reference import oracle_config
from helpers import Golden, assert_close, golden_names, rel_err
from oracle import gin_oracle
from graph_neural_mapping_b200 import engine, lib, ops
from graph_neural_mapping_b200.models import GIN_InfoMaxReg
from graph_neural_mapping_b200.synth import SynthGraph

pytestmark = pytest.mark.gpu
TOL_GRAD = 3e-3


def full_map_mean(model, graphs, cls):
    s = model.compute_saliency_batched(graphs, cls).detach()
    off = np.cumsum([0] + [len(g.g) for g in graphs])
    return torch.stack([s[off[i]:off[i + 1]].mean(0) for i in range(len(graphs))])


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_roi_matches_full_map_mean(name):
    kw, b, n, dense = CONFIGS[name]
    model = make_model(dense if dense is not None else n, **kw)
    graphs = graphs_of(b, n, seed=7, dense_dim=dense)
    roi = model.compute_roi_saliency_batched(graphs, (0, 1))
    assert roi.is_cuda and roi.dtype == torch.float32 and tuple(roi.shape) == (b, 2, dense if dense is not None else n)
    for k, cls in enumerate((0, 1)):
        assert_close(roi[:, k], full_map_mean(model, graphs, cls), 1e-4, "%s class %d" % (name, cls))


def test_ragged_cohort_against_per_graph_saliency():
    d = 400
    model = make_model(d, seed=3)
    g400, = graphs_of(1, 400, seed=11)
    g399, = graphs_of(1, 399, seed=12)
    g37 = SynthGraph(37, 0, 0, torch.eye(37, d))                       # no edges (util.py:17 keeps `0`)
    g1 = SynthGraph(1, 1, 0, torch.eye(1, d))
    cohort = [SynthGraph(len(g.g), g.label, g.edge_mat, torch.eye(len(g.g), d)) for g in (g400, g399)] + [g37, g1]
    roi = model.compute_roi_saliency_batched(cohort, (0, 1))
    for i, x in enumerate(cohort):
        for k, cls in enumerate((0, 1)):
            ref = model.compute_saliency([x], cls).detach().mean(0)
            assert_close(roi[i, k], ref, 1e-4, "graph %d (%d nodes) class %d" % (i, len(x.g), cls))
    assert tuple(model.compute_roi_saliency_batched([], (0, 1)).shape) == (0, 2, d)


def test_isolated_nodes_average_learn_eps():
    """Average pooling divides by the degree: 0/0 = NaN in the forward for a node without neighbours (learn_eps: no self
    loops). The ROI output must be NaN exactly where the full map's node average is."""
    n = 400
    model = make_model(n, eps=True, neigh_pool="average", graph_pool="average", seed=5)
    graphs = []
    for i, g in enumerate(graphs_of(4, n, seed=21)):
        em = g.edge_mat
        if i % 2 == 0:
            cut = torch.tensor([0, 5, 17 + i])
            em = em[:, ~(torch.isin(em[0], cut) | torch.isin(em[1], cut))]
        graphs.append(SynthGraph(n, g.label, em.contiguous(), g.node_features))
    roi = model.compute_roi_saliency_batched(graphs, (0, 1))
    for k, cls in enumerate((0, 1)):
        assert_close(roi[:, k], full_map_mean(model, graphs, cls), 1e-4, "class %d" % cls)


@pytest.mark.parametrize("name", golden_names())
def test_roi_vs_reference_and_oracle(name):
    g = Golden(name)
    c = g.cfg
    model = GIN_InfoMaxReg(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                           c["final_dropout"], c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"], DEV)
    model.load_state_dict(g.state_after_train())
    model = model.to(DEV)
    graphs = g.graphs()
    ocfg = oracle_config(c)
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    for k, v in g.group("saliency/").items():
        gi, cls = int(k[1:k.index("_")]), int(k[-1])
        got = model.compute_roi_saliency_batched([graphs[gi]], (cls,))[0, 0]
        oracle_mean = gin_oracle.saliency(sd, [graphs[gi]], cls, ocfg)[0].mean(0).numpy()
        ref_mean = v.astype(np.float64).mean(0)
        assert_close(got, oracle_mean, TOL_GRAD, "roi vs fp64 oracle " + k)
        own = rel_err(ref_mean, oracle_mean)
        assert_close(got, ref_mean, TOL_GRAD + own, "roi vs reference " + k)


@pytest.fixture(scope="module")
def bench_shape():
    model = make_model(400, seed=1)
    graphs = graphs_of(1024, 400, seed=3)
    model.compute_roi_saliency_batched(graphs, (0,))          # graph store filled, kernels loaded
    return model, graphs


def test_one_forward_serves_both_classes(bench_shape):
    model, graphs = bench_shape
    both, ran2 = launches(lambda: model.compute_roi_saliency_batched(graphs, (0, 1)))
    one0, ran1 = launches(lambda: model.compute_roi_saliency_batched(graphs, (0,)))
    one1, _ = launches(lambda: model.compute_roi_saliency_batched(graphs, (1,)))
    # every kernel here sums in a fixed order (no fp32 atomics on these outputs): bit-identical
    assert torch.equal(both[:, 0], one0[:, 0]) and torch.equal(both[:, 1], one1[:, 0])

    def forward_only():
        bs = model._structure(graphs)
        params = [p.detach() for p in engine.flat_params(model)]
        with torch.no_grad():
            engine.run_forward(model, bs, None, False, False, None, params, engine._dist.SINGLE)
    _, fwd = launches(forward_only)
    assert fwd["linear_tc"] > 0 and fwd["aggregate_tc"] > 0, fwd
    # the second class adds exactly one backward: every family's count grows by (one class) - (the forward)
    for k in ran1:
        assert ran2[k] == ran1[k] + (ran1[k] - fwd[k]), (k, ran1, ran2, fwd)
    assert ran2["linear_tc"] == fwd["linear_tc"], (ran2, fwd)                # the forward's Linear kernels ran once
    assert ran2["segment_colsum"] == 2


def test_launch_counts_against_full_map(bench_shape):
    model, graphs = bench_shape
    _, roi = launches(lambda: model.compute_roi_saliency_batched(graphs, (1,)))
    _, full = launches(lambda: model.compute_saliency_batched(graphs, 1))
    assert roi["aggregate_tc"] == full["aggregate_tc"] - 1, (roi, full)      # no affine aggregation of dz
    assert roi["linear_ffma"] == 0 and full["linear_ffma"] >= 1, (roi, full)  # no [M, 64] -> [M, 400] Linear
    assert roi["segment_colsum"] == 1 and full["segment_colsum"] == 0, (roi, full)
    assert not ops.aggregate_tc_status()


def test_parameter_gradients_untouched():
    model = make_model(400, seed=2)
    graphs = graphs_of(16, 400, seed=4)
    model.compute_saliency([graphs[0]], 1)                    # leaves saliency parameter gradients behind
    model.eps.grad = None
    model.disc.f_k.bias.grad = None
    before = {k: (None if p.grad is None else p.grad.clone()) for k, p in model.named_parameters()}
    assert any(v is None for v in before.values()) and any(v is not None for v in before.values())
    model.train()
    model.compute_roi_saliency_batched(graphs, (0, 1))
    assert not model.training
    for k, p in model.named_parameters():
        if before[k] is None:
            assert p.grad is None, k
        else:
            assert torch.equal(p.grad, before[k]), k


# ---- the kernel alone ------------------------------------------------------------------------------------------------

def _reference(x, node_off, z, coef, rowptr, mode, eps):
    v = x.double()
    if coef is not None:
        v = coef[0].double() * v
        if z is not None:
            v = v + coef[1].double() * z.double() + coef[2].double()
    if rowptr is None:
        w = torch.ones(x.shape[0], dtype=torch.float64, device=x.device)
    else:
        deg = (rowptr[1:] - rowptr[:-1]).double()
        w = (deg > 0).double() if mode == 1 else deg
        if eps is not None:
            w = w + 1.0 + eps.double()
    no = node_off.long()
    gid = torch.repeat_interleave(torch.arange(no.numel() - 1, device=x.device), no[1:] - no[:-1])
    s = torch.zeros(no.numel() - 1, x.shape[1], dtype=torch.float64, device=x.device).index_add_(0, gid, w[:, None] * v)
    return s / (no[1:] - no[:-1]).double().clamp(min=1)[:, None]


@pytest.mark.parametrize("width", [1, 3, 64, 400])
@pytest.mark.parametrize("pad", [0, 3])
def test_kernel_against_torch(width, pad):
    gen = torch.Generator().manual_seed(width * 10 + pad)
    counts = torch.tensor([5, 0, 400, 1, 0, 37, 129, 2])
    node_off = torch.cat([torch.zeros(1, dtype=torch.int64), counts.cumsum(0)]).to(torch.int32).to(DEV)
    m = int(counts.sum())
    deg = torch.randint(0, 9, (m,), generator=gen)
    deg[::17] = 0                                              # isolated rows
    rowptr = torch.cat([torch.zeros(1, dtype=torch.int64), deg.cumsum(0)]).to(torch.int32).to(DEV)
    x, z = strided(m, width, pad, gen), strided(m, width, pad, gen)
    coef = torch.randn(3, width, generator=gen).to(DEV)
    eps = torch.tensor([0.25]).to(DEV)
    b = counts.numel()
    cases = [(None, None, None, 0, None), (None, coef, None, 0, None), (z, coef, rowptr, 0, None), (z, coef, rowptr, 0, eps),
             (None, coef, rowptr, 1, None), (z, coef, rowptr, 1, eps), (None, None, rowptr, 1, eps)]
    for zz, cf, rp, mode, ep in cases:
        out = torch.full((b, width + 2), 7.0, device=DEV)[:, :width]
        ops.segment_weighted_colsum(x, node_off, out, z=zz, coef=cf, rowptr=rp, mode=mode, eps=ep)
        ref = _reference(x, node_off, zz, cf, rp, mode, ep)
        what = "z %s coef %s rowptr %s mode %d eps %s" % (zz is not None, cf is not None, rp is not None, mode, ep is not None)
        assert_close(out, ref.cpu(), 1e-5, what)
        assert bool((out[(counts == 0).to(DEV)] == 0).all()), what + ": empty graphs must give zeros"
    # z = NULL is the eval case cB = cC = 0: bit-identical to passing z with zero cB, cC
    c0 = coef.clone()
    c0[1:] = 0
    a = ops.segment_weighted_colsum(x, node_off, torch.empty(b, width, device=DEV), coef=c0, rowptr=rowptr)
    bb = ops.segment_weighted_colsum(x, node_off, torch.empty(b, width, device=DEV), z=z, coef=c0, rowptr=rowptr)
    assert torch.equal(a, bb)


def test_kernel_argument_checks():
    l = lib.load()
    x = torch.zeros(8, 4, device=DEV)
    out = torch.zeros(2, 4, device=DEV)
    node_off = torch.tensor([0, 4, 8], dtype=torch.int32, device=DEV)
    p = ctypes.c_void_p
    st = p(torch.cuda.current_stream().cuda_stream)

    def call(n_graphs, width, mode=0):
        return l.gnm_segment_weighted_colsum(p(x.data_ptr()), 4, None, 0, None, p(node_off.data_ptr()), n_graphs, width,
                                             None, mode, None, p(out.data_ptr()), 4, st)
    before = ops.launch_counts()
    assert call(-1, 4) == -1 and call(2, -1) == -1 and call(2, 4, mode=2) == -1
    assert call(0, 4) == 0 and call(2, 0) == 0
    assert ops.launch_counts() == before, "an empty or rejected problem must launch nothing"
    assert call(2, 4) == 0
    assert ops.launch_counts()["segment_colsum"] == before["segment_colsum"] + 1
