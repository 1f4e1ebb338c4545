"""ROI occlusion on the GPU: GIN_InfoMaxReg.compute_roi_occlusion_batched (occluded copies as virtual batches of eval
forwards, layer 0 from one real-batch aggregation through gnm_occlusion_expand) against the composed route of existing
code (class_logits on dense copies with one column zeroed), against the fp64 oracle, launch counts, reproducibility, and
the kernel alone against float64 torch."""
import ctypes

import numpy as np
import pytest
import torch

from attribution_cases import CONFIGS, DEV, graphs_of, launches, make_model, strided
from attribution_reference import oracle_config, roi_occlusion as occ_oracle, with_neighbours
from helpers import Golden, assert_close, golden_names
from graph_neural_mapping_b200 import driver, lib, ops
from graph_neural_mapping_b200.models import GIN_InfoMaxReg
from graph_neural_mapping_b200.models import graphcnn as gmod
from graph_neural_mapping_b200.synth import SynthGraph

pytestmark = pytest.mark.gpu
# The score is continuous in the input, so unlike a gradient it cannot jump at a ReLU kink: each class is compared on
# its own max-abs, with the scores' |F_c(X)| / n as floor (the output is a difference of two scores, divided by n).
TOL = 1e-4


def subset(n_cols, k, seed):
    return sorted(np.random.default_rng(seed).choice(n_cols, size=min(k, n_cols), replace=False).tolist())


def composed_route(model, graphs, classes, cols):
    """(F_c(X_i) - F_c(X_i with column d zeroed)) / n_i from driver.class_logits on dense copies, for d in cols[i];
    returns ([B, C, D] with NaN elsewhere, the unoccluded scores [B, C])."""
    d_in = graphs[0].node_features.shape[1]
    copies, where = [], []
    for i, g in enumerate(graphs):
        for d in cols[i]:
            x = g.node_features.clone()
            x[:, d] = 0
            copies.append(SynthGraph(len(g.g), g.label, g.edge_mat, x))
            where.append((i, d))
    f_x = driver.class_logits(model, graphs).double()[:, list(classes)]
    f_d = driver.class_logits(model, copies).double()[:, list(classes)]
    out = torch.full((len(graphs), len(classes), d_in), float("nan"), dtype=torch.float64, device=f_x.device)
    n = torch.tensor([float(len(g.g)) for g in graphs], dtype=torch.float64, device=f_x.device)
    for j, (i, d) in enumerate(where):
        out[i, :, d] = (f_x[i] - f_d[j]) / n[i]
    return out, f_x


def assert_against(out, ref, f_x, graphs, cols, what):
    n = torch.tensor([float(len(g.g)) for g in graphs], dtype=torch.float64, device=f_x.device)
    floor = (f_x.abs() / n[:, None]).nan_to_num(0.0).max(0).values
    for k in range(out.shape[1]):
        got = torch.cat([out[i, k, cols[i]] for i in range(len(graphs))])
        exp = torch.cat([ref[i, k, cols[i]] for i in range(len(graphs))])
        assert_close(got, exp, TOL, "%s class %d" % (what, k), floor=float(floor[k]))


ONEHOT = sorted(k for k, (_, _, _, dense) in CONFIGS.items() if dense is None)


@pytest.mark.parametrize("name", ONEHOT)
def test_matches_composed_route(name):
    kw, b, n, _ = CONFIGS[name]
    model = make_model(n, **kw)
    graphs = graphs_of(b, n, seed=7)
    out = model.compute_roi_occlusion_batched(graphs, (0, 1))
    assert out.is_cuda and out.dtype == torch.float32 and tuple(out.shape) == (b, 2, n)
    few = graphs[:8]                                          # the dense copies: 8 graphs x 32 (16 at N = 1000) ROIs
    cols = [subset(n, 32 if n <= 400 else 16, 100 + i) for i in range(len(few))]
    ref, f_x = composed_route(model, few, (0, 1), cols)
    assert_against(out[:len(few)], ref, f_x, few, cols, name)


@pytest.mark.parametrize("name", golden_names())
def test_against_fp64_oracle(name):
    g = Golden(name)
    c = g.cfg
    model = GIN_InfoMaxReg(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                           c["final_dropout"], c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"], DEV)
    sd = g.state_after_train()
    model.load_state_dict(sd)
    model = model.to(DEV)
    graphs = g.graphs()[:4]
    if name == "tiny_eps_max":
        # nodes without neighbours under max pooling pool the batch's column minimum: rejected, then joined
        with pytest.raises(ValueError, match="without neighbours"):
            model.compute_roi_occlusion_batched(graphs, (0, 1))
        graphs = [with_neighbours(x) for x in graphs]
    d = c["input_dim"]
    cols = list(range(d)) if d < 400 else subset(d, 16, 5)
    out = model.compute_roi_occlusion_batched(graphs, (0, 1)).cpu().double()
    for k in (0, 1):
        ref, f_x = occ_oracle(sd, graphs, k, oracle_config(c), cols=cols)
        n = torch.tensor([float(len(x.g)) for x in graphs], dtype=torch.float64)
        assert_close(out[:, k, cols], ref[:, cols], TOL, "%s class %d" % (name, k), floor=float((f_x.abs() / n).max()))


def test_ragged_cohort():
    d = 400
    model = make_model(d, seed=3)
    g400, = graphs_of(1, 400, seed=11)
    g399, = graphs_of(1, 399, seed=12)
    g37 = SynthGraph(37, 0, 0, torch.eye(37, d))                       # no edges (util.py:17 keeps `0`)
    g1 = SynthGraph(1, 1, 0, torch.eye(1, d))
    cohort = [SynthGraph(len(g.g), g.label, g.edge_mat, torch.eye(len(g.g), d)) for g in (g400, g399)] + [g37, g1]
    out = model.compute_roi_occlusion_batched(cohort, (0, 1))
    cols = [subset(len(x.g), 32, 40 + i) for i, x in enumerate(cohort)]
    ref, f_x = composed_route(model, cohort, (0, 1), cols)
    assert_against(out, ref, f_x, cohort, cols, "ragged")
    for i, x in enumerate(cohort):
        assert bool((out[i, :, len(x.g):] == 0).all()), "graph %d: absent tags must give exactly 0.0" % i
    assert np.array_equal(driver.roi_occlusion(model, cohort, classes=(0, 1)), out.cpu().numpy())
    split = torch.from_numpy(driver.roi_occlusion(model, cohort, classes=(0, 1), batch=3)).to(DEV)
    assert_against(split, out.double(), f_x, cohort, [list(range(d))] * len(cohort), "batch of 3")


def test_isolated_nodes_average_learn_eps():
    """0/0 = NaN in layer 0 for a node without neighbours under average pooling (learn_eps: no self loops): NaN exactly
    where the composed route has NaN, the isolated nodes' own ROIs included, and a graph's row all NaN or none."""
    n = 400
    model = make_model(n, eps=True, neigh_pool="average", graph_pool="average", seed=5)
    graphs = []
    for i, g in enumerate(graphs_of(4, n, seed=21)):
        em = g.edge_mat
        if i % 2 == 0:
            cut = torch.tensor([0, 5, 17 + i], device=em.device)
            em = em[:, ~(torch.isin(em[0], cut) | torch.isin(em[1], cut))]
        graphs.append(SynthGraph(n, g.label, em.contiguous(), g.node_features))
    out = model.compute_roi_occlusion_batched(graphs, (0, 1))
    cols = [[0, 5, 17 + i] + subset(n, 16, 60 + i) for i in range(len(graphs))]
    ref, f_x = composed_route(model, graphs, (0, 1), cols)
    assert_against(out, ref, f_x, graphs, cols, "isolated")
    assert torch.equal(torch.isnan(out).any(2), torch.isnan(out).all(2))


def test_launch_counts_and_reproducibility():
    model = make_model(400, seed=1)
    graphs = graphs_of(40, 400, seed=3)
    model.compute_roi_occlusion_batched(graphs[:1], (0,))
    a, ran = launches(lambda: model.compute_roi_occlusion_batched(graphs, (0, 1)))
    h = model._host_batch(graphs)
    passes = len(gmod.occlusion_passes(h.node_off, model._structure(graphs).tags.cpu().numpy(), 1024))
    assert passes == 16, passes                               # 40 x (400 + 1) virtual graphs, 1024 per pass
    assert ran["occlusion_expand"] == passes, ran
    aggs = ran["aggregate_csr"] + ran["aggregate_mma_sync"] + ran["aggregate_tc"]
    assert aggs == 1 + (model.num_layers - 1) * passes, (aggs, ran)
    assert ran["linear_ffma"] == 0 and ran["linear_tc"] > 0, ran          # no [M, 64] -> [M, 400] Linear
    for fam in ("linear_bwd_ffma", "linear_bwd_dx_tc", "linear_wgrad_tc", "linear_wgrad_ffma", "linear_bwd_onepass_tc",
                "segment_colsum", "ig_expand", "ig_accumulate", "ig_attribute"):
        assert ran[fam] == 0, (fam, ran)
    assert not ops.aggregate_tc_status()
    b = model.compute_roi_occlusion_batched(graphs, (0, 1))
    assert torch.equal(a, b)
    assert torch.equal(a[:, 0], model.compute_roi_occlusion_batched(graphs, (0,))[:, 0])
    assert torch.equal(a[:, 1], model.compute_roi_occlusion_batched(graphs, (1,))[:, 0])


def test_parameter_gradients_untouched():
    model = make_model(400, seed=2)
    graphs = graphs_of(8, 400, seed=4)
    model.compute_saliency([graphs[0]], 1)
    model.eps.grad = None
    before = {k: (None if p.grad is None else p.grad.clone()) for k, p in model.named_parameters()}
    model.train()
    model.compute_roi_occlusion_batched(graphs, (0, 1), occlusions_per_pass=300)
    assert not model.training
    for k, p in model.named_parameters():
        assert (p.grad is None) == (before[k] is None) and (p.grad is None or torch.equal(p.grad, before[k])), k


# ---- the kernel alone ------------------------------------------------------------------------------------------------

COUNTS = [5, 0, 400, 1, 37, 129, 2]
D_TAGS = 450


def _real_batch(gen, self_loops):
    """Random symmetric graphs (isolated nodes included) with duplicate tags: dense adjacency, CSR with global ids."""
    m = sum(COUNTS)
    adj = torch.zeros(m, m, dtype=torch.float64)
    off = np.cumsum([0] + COUNTS)
    for g, n in enumerate(COUNTS):
        a = (torch.rand(n, n, generator=gen) < 0.1).double()
        a = torch.triu(a, 1)
        a = a + a.t()
        if self_loops:
            a = a + torch.eye(n, dtype=torch.float64)
        adj[off[g]:off[g + 1], off[g]:off[g + 1]] = a
    adj[off[2] + 7] = 0                                       # an isolated node in the 400-node graph
    adj[:, off[2] + 7] = 0
    rows, cols = adj.nonzero(as_tuple=True)
    rowptr = torch.zeros(m + 1, dtype=torch.int64)
    rowptr[1:] = torch.bincount(rows, minlength=m).cumsum(0)
    tags = torch.randint(0, D_TAGS, (m,), generator=gen)
    tags[off[2] + 10:off[2] + 20] = 3                         # duplicate tags
    node_off = torch.tensor(off, dtype=torch.int32)
    return adj, rowptr.to(torch.int32), cols.to(torch.int32), tags.to(torch.int32), node_off


@pytest.mark.parametrize("width", [3, 64])
@pytest.mark.parametrize("pad", [0, 3])
@pytest.mark.parametrize("mode,learn_eps", [(0, False), (0, True), (1, True)])
def test_kernel_against_torch(width, pad, mode, learn_eps):
    gen = torch.Generator().manual_seed(width * 10 + pad + 100 * mode + learn_eps)
    adj, rowptr, colidx, tags, node_off = _real_batch(gen, not learn_eps)
    m = adj.shape[0]
    off = node_off.long().tolist()
    # virtual graphs: per real graph a baseline, every present tag, and an absent tag; v_tag 3 twice in graph 2
    v_graph, v_tag = [], []
    for g in range(len(COUNTS)):
        present = sorted(set(tags[off[g]:off[g + 1]].tolist()))
        absent = next(t for t in range(D_TAGS) if t not in present)
        for t in [-1] + present + [absent]:
            v_graph.append(g)
            v_tag.append(t)
    v_node_off = np.cumsum([0] + [COUNTS[g] for g in v_graph])
    p = strided(m, width, pad, gen)
    w1t = strided(D_TAGS, width, pad, gen)
    bias = torch.randn(width, generator=gen).to(DEV)
    eps = torch.tensor([0.3]).to(DEV) if learn_eps else None
    z = strided(int(v_node_off[-1]), width, pad, gen)
    to_d = lambda t: t.to(DEV)
    ops.occlusion_expand(p, bias, w1t, to_d(rowptr), to_d(colidx), to_d(tags), to_d(node_off), max(COUNTS),
                         to_d(torch.tensor(v_graph, dtype=torch.int32)), to_d(torch.tensor(v_tag, dtype=torch.int32)),
                         to_d(torch.tensor(v_node_off, dtype=torch.int32)), mode, eps, z)
    onehot = torch.nn.functional.one_hot(tags.long(), D_TAGS).double()
    counts = adj @ onehot                                     # [M, D]: #{n in row m : tags[n] = d}
    deg = adj.sum(1, keepdim=True)
    coef = torch.where(counts != 0, counts / deg if mode == 1 else counts, torch.zeros_like(counts))
    if learn_eps:
        coef = coef + (1.0 + 0.3) * onehot
    base32 = (p + bias).cpu()
    pc, wc = p.double().cpu() + bias.double().cpu(), w1t.double().cpu()
    zc = z.cpu()
    for v, (g, t) in enumerate(zip(v_graph, v_tag)):
        r0, r1 = off[g], off[g + 1]
        got = zc[v_node_off[v]:v_node_off[v + 1]]
        if t < 0:
            assert torch.equal(got, base32[r0:r1]), "baseline copy %d: not exactly p + bias" % v
            continue
        c = coef[r0:r1, t]
        ref = pc[r0:r1] - c[:, None] * wc[t]
        assert_close(got, ref, 1e-6, "copy %d (graph %d, tag %d)" % (v, g, t))
        same = c == 0
        assert torch.equal(got[same], base32[r0:r1][same]), "copy %d: unaffected rows not exactly p + bias" % v


def test_kernel_argument_checks():
    l = lib.load()
    p = ctypes.c_void_p
    x = torch.zeros(16, 4, device=DEV)
    i32 = torch.zeros(16, dtype=torch.int32, device=DEV)
    xp, ip = p(x.data_ptr()), p(i32.data_ptr())
    st = p(torch.cuda.current_stream().cuda_stream)

    def call(n_max=4, n_virtual=2, width=4, mode=0):
        return l.gnm_occlusion_expand(xp, 4, None, xp, 4, 4, ip, ip, ip, ip, 2, n_max, ip, ip, ip, n_virtual, width, mode,
                                      None, xp, 4, st)
    before = ops.launch_counts()
    assert call(n_virtual=-1) == -1 and call(mode=3) == -1
    assert call(n_virtual=0) == 0 and call(width=0) == 0
    assert call(n_max=5000) == -2                             # GNM_ERR_TOO_LARGE
    assert ops.launch_counts() == before, "an empty or rejected problem must launch nothing"
    with pytest.raises(RuntimeError, match="gnm_occlusion_expand"):
        ops.occlusion_expand(x, None, x, i32, i32, i32, i32[:3], 5000, i32[:2], i32[:2], i32[:3], 0, None, x)
