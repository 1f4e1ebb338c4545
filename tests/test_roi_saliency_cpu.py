"""Host logic of ROI saliency on CPU: GIN_InfoMaxReg.compute_roi_saliency_batched / driver.roi_saliency over the CPU
stand-in kernels (tests/emul_ops.py). Checks the node averages against the reference's saliency maps in the golden
fixtures, the one-forward / many-backward reuse, and that no parameter gradient is written."""
import numpy as np
import pytest
import torch

from helpers import Golden, assert_close, build_model, golden_names, use_cpu_stand_in
from graph_neural_mapping_b200 import driver, engine
from graph_neural_mapping_b200.synth import SynthGraph

NAMES = [n for n in golden_names() if Golden(n).cfg["N"] < 400]     # the dense CPU stand-in is too slow at N = 400
TOL_GRAD = 2e-3


@pytest.fixture(autouse=True)
def cpu_backend(monkeypatch):
    use_cpu_stand_in(monkeypatch)


@pytest.mark.parametrize("name", NAMES)
def test_roi_matches_reference_saliency_mean(name):
    g = Golden(name)
    model = build_model(g, g.state_after_train())
    graphs = g.graphs()
    maxpool = g.cfg["neighbor_pooling_type"] == "max"
    # under max pooling the dummy row is a batch-wide minimum (graphcnn.py:140): the reference's maps are per graph
    roi = None if maxpool else model.compute_roi_saliency_batched(graphs[:2], (0, 1))
    for k, v in g.group("saliency/").items():
        gi, cls = int(k[1:k.index("_")]), int(k[-1])
        got = model.compute_roi_saliency_batched([graphs[gi]], (cls,))[0, 0] if maxpool else roi[gi, cls]
        assert_close(got, v.mean(0), TOL_GRAD, "roi " + k)


@pytest.mark.parametrize("name", ["tiny_eps_avg", "tiny_mlp3", "tiny_noeps_max", "mid_eps_sum_h64"])
def test_one_forward_serves_every_class(name, monkeypatch):
    g = Golden(name)
    model = build_model(g, g.state_after_train())
    graphs = g.graphs()[:2] if g.cfg["neighbor_pooling_type"] != "max" else g.graphs()[:1]
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
    both = model.compute_roi_saliency_batched(graphs, (0, 1))
    assert calls == {"fwd": 1, "bwd": 2}
    assert tuple(both.shape) == (len(graphs), 2, g.cfg["input_dim"])
    assert torch.equal(both[:, 0], model.compute_roi_saliency_batched(graphs, (0,))[:, 0])
    assert torch.equal(both[:, 1], model.compute_roi_saliency_batched(graphs, [1])[:, 0])
    for k, p in model.named_parameters():
        assert (p.grad is None) == (before[k] is None) and (p.grad is None or torch.equal(p.grad, before[k])), k
    assert not model.training
    # against the full map of the same code path, averaged per graph
    n0 = len(graphs[0].g)
    for k, cls in enumerate((0, 1)):
        full = model.compute_saliency_batched(graphs, cls).detach()
        assert_close(both[0, k], full[:n0].mean(0), 1e-5, "class %d g0" % cls)
        if len(graphs) > 1:
            assert_close(both[1, k], full[n0:].mean(0), 1e-5, "class %d g1" % cls)


def test_ragged_cohort_and_driver():
    # without learn_eps every node keeps its self loop: the dense CPU stand-in would spread an isolated node's forward NaN
    # (average pooling, 0/0) over the whole batch, which the CUDA kernels do not (covered on the GPU)
    g = Golden("tiny_noeps_avg")
    model = build_model(g, g.state_after_train())
    src = g.graphs()
    d = g.cfg["input_dim"]
    # graphs of 16, 7 and 1 nodes, the last without edges
    small = SynthGraph(7, 0, src[1].edge_mat[:, (src[1].edge_mat < 7).all(0)], torch.eye(7, d))
    lone = SynthGraph(1, 1, 0, torch.eye(1, d))
    cohort = [src[0], small, lone]
    roi = driver.roi_saliency(model, cohort, classes=(1, 0), batch=2)
    assert roi.dtype == np.float32 and roi.shape == (3, 2, d)
    for i, x in enumerate(cohort):
        for k, cls in enumerate((1, 0)):
            ref = model.compute_saliency([x], cls).detach().mean(0)
            assert_close(roi[i, k], ref, 1e-5, "graph %d class %d" % (i, cls))
    assert driver.roi_saliency(model, [], classes=(0, 1)).shape == (0, 2, d)
