"""Host logic of integrated gradients on CPU: GIN_InfoMaxReg.compute_integrated_gradients_batched /
driver.integrated_gradients over the CPU stand-in kernels (tests/emul_ops.py). Checks the attributions and the
completeness gap against plain autograd on the fp64 oracle (tests/attribution_reference.py), the virtual-batch plumbing
(one forward per pass, one backward per class and pass, chunking), the argument errors, and that the new entry points
check their arguments without a GPU."""
import numpy as np
import pytest
import torch

from attribution_reference import integrated_gradients as ig_oracle, oracle_config
from helpers import Golden, assert_close, build_model, use_cpu_stand_in
from graph_neural_mapping_b200 import driver, engine, lib
from graph_neural_mapping_b200.synth import SynthGraph

NAMES = ["tiny_eps_sum", "tiny_noeps_sum", "tiny_eps_avg", "tiny_noeps_avg", "tiny_mlp1", "tiny_mlp3", "mid_eps_sum_h64"]
TOL_GRAD = 2e-3


@pytest.fixture(autouse=True)
def cpu_backend(monkeypatch):
    use_cpu_stand_in(monkeypatch)


@pytest.mark.parametrize("name", NAMES)
def test_matches_oracle(name):
    g = Golden(name)
    sd = g.state_after_train()
    model = build_model(g, sd)
    graphs = g.graphs()[:3]
    out, delta = model.compute_integrated_gradients_batched(graphs, (0, 1), steps=8, return_delta=True)
    assert tuple(out.shape) == (len(graphs), 2, g.cfg["input_dim"]) and tuple(delta.shape) == (len(graphs), 2)
    for k in (0, 1):
        ref, ref_delta, f_x, f_0 = ig_oracle(sd, graphs, k, oracle_config(g.cfg), 8)
        assert_close(out[:, k], ref, TOL_GRAD, "%s class %d" % (name, k))
        # the gap is a small difference of two scores: compare on their scale
        scale = float((f_x.abs() + f_0.abs()).max())
        assert_close(delta[:, k], ref_delta, TOL_GRAD, "%s delta class %d" % (name, k), floor=scale)


@pytest.mark.parametrize("name", ["tiny_noeps_sum", "tiny_eps_avg", "mid_eps_sum_h64"])
def test_oracle_gap_closes(name):
    """Completeness of the midpoint rule itself: at S = 512 the oracle's gap is below 2e-3 of |F(X)| + |F(0)|."""
    g = Golden(name)
    _, delta, f_x, f_0 = ig_oracle(g.state_after_train(), g.graphs()[:2], 1, oracle_config(g.cfg), 512)
    assert float((delta.abs() / (f_x.abs() + f_0.abs())).max()) < 2e-3


@pytest.mark.parametrize("name", ["tiny_eps_avg", "tiny_mlp3", "mid_eps_sum_h64"])
def test_passes_chunks_and_grads(name, monkeypatch):
    g = Golden(name)
    model = build_model(g, g.state_after_train())
    graphs = g.graphs()[:3]
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
    one = model.compute_integrated_gradients_batched(graphs, (0, 1), steps=6)
    assert calls == {"fwd": 1, "bwd": 2}              # one pass: every graph's 6 points in one virtual batch
    for k, p in model.named_parameters():
        assert (p.grad is None) == (before[k] is None) and (p.grad is None or torch.equal(p.grad, before[k])), k
    assert not model.training
    # 4 points per pass < steps: one graph per chunk, its points over two passes (4 + 2) that accumulate
    calls.update(fwd=0, bwd=0)
    split = model.compute_integrated_gradients_batched(graphs, (0, 1), steps=6, points_per_pass=4)
    assert calls == {"fwd": 3 * 2, "bwd": 3 * 2 * 2}
    assert_close(split, one, 1e-6, "points over several passes")
    # 13 points per pass: two graphs per chunk, chunks of 2 + 1 graphs
    calls.update(fwd=0, bwd=0)
    two = model.compute_integrated_gradients_batched(graphs, (0, 1), steps=6, points_per_pass=13)
    assert calls == {"fwd": 2, "bwd": 4}
    assert_close(two, one, 1e-6, "graphs over several chunks")
    assert torch.equal(one[:, 1], model.compute_integrated_gradients_batched(graphs, [1], steps=6)[:, 0])


def test_ragged_cohort_and_driver():
    g = Golden("tiny_noeps_avg")
    sd = g.state_after_train()
    model = build_model(g, sd)
    src = g.graphs()
    d = g.cfg["input_dim"]
    # graphs of 16, 7 and 1 nodes, the last without edges; the 7-node graph carries a duplicate tag
    feats = torch.eye(7, d)
    feats[6] = feats[2]
    small = SynthGraph(7, 0, src[1].edge_mat[:, (src[1].edge_mat < 7).all(0)], feats)
    lone = SynthGraph(1, 1, torch.zeros(2, 0, dtype=torch.int64), torch.eye(1, d))
    cohort = [src[0], small, lone]
    out, delta = driver.integrated_gradients(model, cohort, classes=(1, 0), steps=5, batch=2, return_delta=True)
    assert out.dtype == np.float32 and out.shape == (3, 2, d) and delta.shape == (3, 2)
    cfg = oracle_config(g.cfg)
    for i, x in enumerate(cohort):
        for k, cls in enumerate((1, 0)):
            ref, ref_delta, f_x, f_0 = ig_oracle(sd, [x], cls, cfg, 5)
            assert_close(out[i, k], ref[0], TOL_GRAD, "graph %d class %d" % (i, cls))
            assert abs(float(delta[i, k]) - float(ref_delta[0])) <= TOL_GRAD * float(f_x.abs() + f_0.abs())
    assert np.array_equal(out, driver.integrated_gradients(model, cohort, classes=(1, 0), steps=5))
    assert driver.integrated_gradients(model, [], classes=(0, 1)).shape == (0, 2, d)
    e, ed = model.compute_integrated_gradients_batched([], (0, 1), return_delta=True)
    assert tuple(e.shape) == (0, 2, d) and tuple(ed.shape) == (0, 2)


def test_rejects_what_it_cannot_attribute():
    g = Golden("tiny_eps_sum")
    model = build_model(g)
    graphs = g.graphs()[:2]
    with pytest.raises(ValueError, match="classes"):
        model.compute_integrated_gradients_batched(graphs, (0, 2))
    with pytest.raises(ValueError, match="steps"):
        model.compute_integrated_gradients_batched(graphs, (0,), steps=0)
    dense = SynthGraph(12, 0, graphs[0].edge_mat, torch.rand(12, g.cfg["input_dim"]))
    with pytest.raises(ValueError, match="one-hot"):
        model.compute_integrated_gradients_batched([graphs[0], dense], (0,))
    gm = Golden("tiny_eps_max")
    with pytest.raises(ValueError, match="max pooling"):
        build_model(gm).compute_integrated_gradients_batched(gm.graphs()[:1], (0,))


def test_argument_checks_need_no_gpu():
    """The new entry points validate arguments before touching the device: negative sizes give GNM_ERR_BAD_ARG, empty
    problems GNM_OK without a launch."""
    l = lib.load()
    assert l.gnm_ig_expand(None, 0, None, None, None, -1, 0, 1, 4, None, 4, None) == -1
    assert l.gnm_ig_expand(None, 0, None, None, None, 2, 0, 1, -4, None, 4, None) == -1
    assert l.gnm_ig_expand(None, 0, None, None, None, 0, 0, 3, 4, None, 4, None) == 0
    assert l.gnm_ig_expand(None, 0, None, None, None, 2, 10, 0, 4, None, 4, None) == 0
    assert l.gnm_ig_accumulate(None, 0, None, None, 2, 10, -1, 4, 1.0, 0, None, 4, None) == -1
    assert l.gnm_ig_accumulate(None, 0, None, None, 2, 0, 3, 4, 1.0, 0, None, 4, None) == 0
    assert l.gnm_ig_accumulate(None, 0, None, None, 2, 10, 3, 0, 1.0, 1, None, 4, None) == 0
    assert l.gnm_ig_attribute(None, 0, None, 0, 5, None, None, -1, 4, None, 5, None) == -1
    assert l.gnm_ig_attribute(None, 0, None, 0, -5, None, None, 2, 4, None, 5, None) == -1
    assert l.gnm_ig_attribute(None, 0, None, 0, 5, None, None, 0, 4, None, 5, None) == 0
