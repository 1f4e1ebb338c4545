"""Host logic of ROI occlusion on CPU: GIN_InfoMaxReg.compute_roi_occlusion_batched / driver.roi_occlusion over the CPU
stand-in kernels (tests/emul_ops.py). Checks the output against the fp64 oracle (tests/attribution_reference.py), the
pass planning (graphs split over passes, several graphs per pass, one forward per pass), the argument errors, and that
the new entry point checks its arguments without a GPU."""
import numpy as np
import pytest
import torch

from attribution_reference import oracle_config, roi_occlusion as occ_oracle, with_neighbours
from helpers import Golden, assert_close, build_model, use_cpu_stand_in
from graph_neural_mapping_b200 import driver, engine, lib
from graph_neural_mapping_b200.models import graphcnn as gmod
from graph_neural_mapping_b200.synth import SynthGraph

NAMES = ["tiny_eps_sum", "tiny_noeps_sum", "tiny_eps_avg", "tiny_noeps_avg", "tiny_eps_max", "tiny_noeps_max",
         "tiny_mlp1", "tiny_mlp3", "mid_eps_sum_h64"]
TOL = 1e-4


@pytest.fixture(autouse=True)
def cpu_backend(monkeypatch):
    use_cpu_stand_in(monkeypatch)


def assert_matches(out, ref, f_x, n, what):
    """Per class on its own max-abs, with the scores' |F_c(X)| / n as floor (the output is a difference of scores)."""
    assert_close(out, ref, TOL, what, floor=float((f_x.abs() / n).max()))


@pytest.mark.parametrize("name", NAMES)
def test_matches_oracle(name):
    g = Golden(name)
    sd = g.state_after_train()
    model = build_model(g, sd)
    graphs = g.graphs()
    if name == "tiny_eps_max":
        # every graph has a node without neighbours (learn_eps: no self loop): max pooling gives it the column minimum
        # of h over the forward's whole batch, so the occluded score of a graph is not its own
        with pytest.raises(ValueError, match="without neighbours"):
            model.compute_roi_occlusion_batched(graphs, (0, 1))
        # the same graphs with those nodes joined to a neighbour
        graphs = [with_neighbours(x) for x in graphs]
    out = model.compute_roi_occlusion_batched(graphs, (0, 1))
    assert tuple(out.shape) == (len(graphs), 2, g.cfg["input_dim"]) and out.dtype == torch.float32
    n = torch.tensor([float(len(x.g)) for x in graphs], dtype=torch.float64)
    for k in (0, 1):
        ref, f_x = occ_oracle(sd, graphs, k, oracle_config(g.cfg))
        assert_matches(out[:, k], ref, f_x, n, "%s class %d" % (name, k))


def test_pass_planning():
    node_off = np.array([0, 3, 3, 8, 9], dtype=np.int32)
    tags = np.array([2, 0, 2, 4, 1, 3, 1, 0, 7], dtype=np.int32)      # graph 0: tags {0, 2}; graph 1 empty
    plan = gmod.occlusion_passes(node_off, tags, 1024)
    assert len(plan) == 1
    assert plan[0][0].tolist() == [0, 0, 0, 2, 2, 2, 2, 2, 3, 3]
    assert plan[0][1].tolist() == [-1, 0, 2, -1, 0, 1, 3, 4, -1, 7]
    # a graph's tags split over passes, each pass with its own baseline; at most 4 virtual graphs per pass
    plan = gmod.occlusion_passes(node_off, tags, 4)
    assert [p[0].tolist() for p in plan] == [[0, 0, 0], [2, 2, 2, 2], [2, 2, 3, 3]]
    assert [p[1].tolist() for p in plan] == [[-1, 0, 2], [-1, 0, 1, 3], [-1, 4, -1, 7]]
    # 1 (and 2): one baseline and one occluded copy per pass
    for cap in (1, 2):
        plan = gmod.occlusion_passes(node_off, tags, cap)
        assert [p[1].tolist() for p in plan] == [[-1, 0], [-1, 2], [-1, 0], [-1, 1], [-1, 3], [-1, 4], [-1, 7]]
        assert [p[0].tolist() for p in plan] == [[0, 0], [0, 0], [2, 2], [2, 2], [2, 2], [2, 2], [3, 3]]


@pytest.mark.parametrize("name", ["tiny_eps_avg", "tiny_noeps_max", "mid_eps_sum_h64"])
def test_passes_and_grads(name, monkeypatch):
    g = Golden(name)
    model = build_model(g, g.state_after_train())
    graphs = g.graphs()[:3]
    d = g.cfg["input_dim"]
    for p in model.parameters():
        p.grad = None
    model.eps.grad = torch.full_like(model.eps, 7.0)
    before = {k: (None if p.grad is None else p.grad.clone()) for k, p in model.named_parameters()}
    calls = {"fwd": 0, "bwd": 0}
    real_fwd, real_bwd = engine.run_forward, engine.run_backward

    def fwd(*a, **kw):
        calls["fwd"] += 1
        return real_fwd(*a, **kw)

    def bwd(*a, **kw):
        calls["bwd"] += 1
        return real_bwd(*a, **kw)
    monkeypatch.setattr(engine, "run_forward", fwd)
    monkeypatch.setattr(engine, "run_backward", bwd)
    model.train()
    one = model.compute_roi_occlusion_batched(graphs, (0, 1))
    assert calls == {"fwd": 1, "bwd": 0}                 # every graph's copies in one virtual batch, no backward
    for k, p in model.named_parameters():
        assert (p.grad is None) == (before[k] is None) and (p.grad is None or torch.equal(p.grad, before[k])), k
    assert not model.training
    n_present = [len(set(x.node_features.argmax(1).tolist())) for x in graphs]
    n = torch.tensor([float(len(x.g)) for x in graphs], dtype=torch.float64)
    f_x = [occ_oracle(g.state_after_train(), graphs, k, oracle_config(g.cfg), cols=[])[1] for k in (0, 1)]
    for per, expect in ((d // 2 + 1, None), (2 * d + 5, 2), (1, sum(n_present))):
        calls.update(fwd=0)
        res = model.compute_roi_occlusion_batched(graphs, (0, 1), occlusions_per_pass=per)
        if expect is not None:
            assert calls["fwd"] == expect, (per, calls)
        else:
            assert calls["fwd"] > len(graphs), (per, calls)          # every graph's ROIs split over two passes
        for k in (0, 1):
            # other batch compositions round the scores differently (the stand-in's dense products change shape)
            assert_matches(res[:, k], one[:, k], f_x[k], n, "occlusions_per_pass %d class %d" % (per, k))
    assert torch.equal(one[:, 1], model.compute_roi_occlusion_batched(graphs, [1])[:, 0])


def test_ragged_cohort_and_driver():
    g = Golden("tiny_noeps_avg")
    sd = g.state_after_train()
    model = build_model(g, sd)
    src = g.graphs()
    d = g.cfg["input_dim"]
    # graphs of 16, 7 and 1 nodes, the last without edges; the 7-node graph carries a duplicate tag and lacks tags 7..15
    feats = torch.eye(7, d)
    feats[6] = feats[2]
    small = SynthGraph(7, 0, src[1].edge_mat[:, (src[1].edge_mat < 7).all(0)], feats)
    lone = SynthGraph(1, 1, torch.zeros(2, 0, dtype=torch.int64), torch.eye(1, d))
    cohort = [src[0], small, lone]
    out = driver.roi_occlusion(model, cohort, classes=(1, 0), batch=2)
    assert out.dtype == np.float32 and out.shape == (3, 2, d)
    cfg = oracle_config(g.cfg)
    for i, x in enumerate(cohort):
        present = sorted(set(x.node_features.argmax(1).tolist()))
        absent = [c for c in range(d) if c not in present]
        for k, cls in enumerate((1, 0)):
            ref, f_x = occ_oracle(sd, [x], cls, cfg, cols=present)
            assert_close(out[i, k, present], ref[0, present], TOL, "graph %d class %d" % (i, cls),
                         floor=float(f_x.abs().max()) / len(x.g))
            assert (out[i, k, absent] == 0.0).all(), "absent tags must give exactly 0"
    assert np.array_equal(out, driver.roi_occlusion(model, cohort, classes=(1, 0), batch=2))
    assert driver.roi_occlusion(model, [], classes=(0, 1)).shape == (0, 2, d)
    assert tuple(model.compute_roi_occlusion_batched(src[:2], ()).shape) == (2, 0, d)


def test_rejects_what_it_cannot_occlude():
    g = Golden("tiny_eps_sum")
    model = build_model(g)
    graphs = g.graphs()[:2]
    with pytest.raises(ValueError, match="classes"):
        model.compute_roi_occlusion_batched(graphs, (0, 2))
    with pytest.raises(ValueError, match="occlusions_per_pass"):
        model.compute_roi_occlusion_batched(graphs, (0,), occlusions_per_pass=0)
    dense = SynthGraph(12, 0, graphs[0].edge_mat, torch.rand(12, g.cfg["input_dim"]))
    with pytest.raises(ValueError, match="one-hot"):
        model.compute_roi_occlusion_batched([graphs[0], dense], (0,))
    no_stats = build_model(g)
    no_stats.batch_norms[0].track_running_stats = False
    with pytest.raises(ValueError, match="running statistics"):
        no_stats.compute_roi_occlusion_batched(graphs, (0,))
    gm = Golden("tiny_noeps_max")
    x = gm.graphs()[0]
    feats = x.node_features.clone()
    feats[3] = feats[5]                                            # a repeated tag: layer 0's max is not its sum
    with pytest.raises(ValueError, match="max neighbour pooling"):
        build_model(gm).compute_roi_occlusion_batched([SynthGraph(len(x.g), 0, x.edge_mat, feats)], (0,))


def test_argument_checks_need_no_gpu():
    """The new entry point validates arguments before touching the device: negative sizes give GNM_ERR_BAD_ARG, empty
    problems GNM_OK without a launch."""
    l = lib.load()
    nul = [None] * 7

    def call(n_table_rows=4, n_graphs=2, n_max=5, n_virtual=3, width=4, mode=0):
        return l.gnm_occlusion_expand(None, 4, None, None, 4, n_table_rows, *nul[:4], n_graphs, n_max, *nul[:3],
                                      n_virtual, width, mode, None, None, 4, None)
    assert call(n_table_rows=-1) == -1 and call(n_graphs=-1) == -1 and call(n_max=-1) == -1
    assert call(n_virtual=-1) == -1 and call(width=-4) == -1 and call(mode=2) == -1
    assert call(n_virtual=0) == 0 and call(width=0) == 0 and call(n_max=0) == 0
