"""The training step's one-pass DGI scorer (gnm_dgi_score_train: scores + BCEWithLogits + the scorer's backward from one
read of n_f) against the three calls it replaces - gnm_dgi_score_fwd, gnm_bce_logits, gnm_dgi_score_bwd - and a whole
driver.Trainer step against the same step with the scorer declined (the three-call path)."""
import numpy as np
import pytest
import torch

from helpers import Golden, SEED0, assert_close, grad_floor
from graph_neural_mapping_b200 import ops
from graph_neural_mapping_b200.models import GIN_InfoMaxReg

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _inputs(L, f, counts, seed):
    g = torch.Generator().manual_seed(seed)
    b = len(counts)
    m = int(sum(counts))
    h_all = torch.randn(L, m, f, generator=g).to(DEV)
    u = (0.2 * torch.randn(b, L * f, generator=g)).to(DEV)
    bias = torch.tensor([0.3], device=DEV)
    perm = torch.randperm(b, generator=g).to(torch.int32).to(DEV)
    no = torch.from_numpy(np.cumsum([0] + list(counts)).astype(np.int32)).to(DEV)
    return h_all, u, bias, perm, no, b, m


def _three_calls(h_all, u, table, perm, no, b, m, bias, w):
    out = torch.empty(2 * m, 1, device=DEV)
    ops.dgi_score_fwd(h_all, u, table, perm, no, b, bias, out)
    loss = torch.zeros(1, dtype=torch.float64, device=DEV)
    dd = torch.empty(2 * m, device=DEV)
    ops.bce_logits(out.view(-1), m, w, w, loss, dd)
    du, s2 = torch.empty(b, u.shape[1], device=DEV), torch.empty(b, device=DEV)
    db = torch.zeros(1, dtype=torch.float64, device=DEV)
    ops.dgi_score_bwd(h_all, dd, table, perm, no, b, du, s2, db)
    return out, dd[:m], du, s2, db, loss


RAGGED = [0, 1, 416, 37, 129, 400, 63, 255, 2, 300, 65, 191, 7, 411]


@pytest.mark.parametrize("L,counts", [(5, [400] * 1024), (5, [400] * 3), (5, RAGGED), (3, RAGGED), (4, [129, 1, 64]),
                                      (2, [5, 0, 17]), (1, [33, 8])])
def test_one_pass_scorer_matches_the_three_calls(L, counts):
    h_all, u, bias, perm, no, b, m = _inputs(L, 64, counts, seed=L * 1000 + len(counts))
    table = ops.gather_nf_rows(h_all, b)
    w = 0.05 / (2.0 * m)
    out0, ds0, du0, s20, db0, loss0 = _three_calls(h_all, u, table, perm, no, b, m, bias, w)
    out = torch.empty(2 * m, 1, device=DEV)
    ds, du, s2 = torch.empty(m, device=DEV), torch.empty(b, L * 64, device=DEV), torch.empty(b, device=DEV)
    db, loss = torch.zeros(1, dtype=torch.float64, device=DEV), torch.zeros(1, dtype=torch.float64, device=DEV)
    assert ops.dgi_score_train(h_all, u, table, perm, no, b, bias, w, w, out, ds, du, s2, db, loss)
    # same rows per thread and the same operation order as the three kernels: the scores and their gradient are
    # bit-identical; the negatives' gradient is formed once per graph instead of once per row and may round 1 ulp
    # apart, which reaches s2 (a sum of those) and du through s2 * neg_table
    assert torch.equal(out, out0)
    assert torch.equal(ds, ds0)
    assert_close(s2, s20, 1e-5, "s2")
    assert_close(du, du0, 1e-5, "du")
    # d_bias = sum of the positive and negative gradients, which nearly cancel: compared on the scale of its terms
    assert float((db - db0).abs()) <= 1e-6 * float(ds.abs().sum() + s2.abs().sum())
    # the same fp32 loss terms, summed in double in another order
    assert_close(loss, loss0, 1e-9, "loss")
    # and against torch's BCEWithLogitsLoss on the scores (main.py:32-34); the kernels form each term in fp32
    y = torch.cat([torch.ones(m, 1), torch.zeros(m, 1)], 0).to(DEV)
    ref = torch.nn.functional.binary_cross_entropy_with_logits(out.double(), y.double(), reduction="sum") * w
    assert_close(loss, ref.view(1), 1e-6, "loss vs torch")


def test_one_pass_scorer_declines_other_widths():
    h_all, u, bias, perm, no, b, m = _inputs(3, 32, [10, 12, 9], seed=3)
    table = ops.gather_nf_rows(h_all, b)
    out = torch.empty(2 * m, 1, device=DEV)
    ds, du, s2 = torch.empty(m, device=DEV), torch.empty(b, 96, device=DEV), torch.empty(b, device=DEV)
    db, loss = torch.zeros(1, dtype=torch.float64, device=DEV), torch.zeros(1, dtype=torch.float64, device=DEV)
    before = ops.kernels_recorded()
    assert ops.dgi_score_train(h_all, u, table, perm, no, b, bias, 1e-3, 1e-3, out, ds, du, s2, db, loss) is False
    assert ops.kernels_recorded() == before


def _build_model(g):
    c = g.cfg
    m = GIN_InfoMaxReg(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                       0.0, c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"], torch.device(DEV))
    m.load_state_dict(g.state_dict())
    return m.to(DEV).train()


def _counting(monkeypatch, names, calls):
    for n in names:
        fn = getattr(ops, n)

        def wrapped(*a, _fn=fn, _n=n, **k):
            calls[_n] = calls.get(_n, 0) + 1
            return _fn(*a, **k)
        monkeypatch.setattr(ops, n, wrapped)


@pytest.mark.parametrize("name", ["schaefer400_b16_noeps", "schaefer400_b16_eps", "mid_eps_sum_h64"])
def test_trainer_step_with_one_pass_scorer_matches_three_call_step(name, monkeypatch):
    """One eager Trainer step from the fixture's state, with the one-pass scorer and with it declined: loss, every
    gradient and the BatchNorm buffers, each tensor on its own max-abs."""
    from graph_neural_mapping_b200.driver import Trainer
    g = Golden(name)
    graphs = g.graphs()
    runs = []
    for one_pass in (False, True):
        with monkeypatch.context() as mp:
            calls = {}
            if not one_pass:
                mp.setattr(ops, "dgi_score_train", lambda *a, **k: False)
            _counting(mp, ["dgi_score_train", "dgi_score_fwd", "dgi_score_bwd", "bce_logits", "bn_relu_readout"], calls)
            model = _build_model(g)
            tr = Trainer(model, lr=0.005, beta=g.cfg["beta"])
            np.random.seed(4242 + SEED0[name])
            loss = float(tr.step(graphs))
            torch.cuda.synchronize()
            grads = {k: p.grad.detach().clone() for k, p in model.named_parameters() if p.grad is not None}
            bufs = {k: v.detach().clone() for k, v in model.state_dict().items() if "running" in k}
            tr.finish()
            runs.append((loss, grads, bufs, calls))
    (loss0, g0, b0, c0), (loss1, g1, b1, c1) = runs
    assert c0.get("dgi_score_bwd") == c0.get("bce_logits") == c0.get("dgi_score_fwd") == 1, c0
    assert c1.get("dgi_score_train") == 1 and "dgi_score_bwd" not in c1 and "bce_logits" not in c1 \
        and "dgi_score_fwd" not in c1, c1
    assert c1.get("bn_relu_readout") == c0.get("bn_relu_readout"), (c0, c1)
    assert_close(np.array(loss1), np.array(loss0), 1e-6, "loss")
    assert set(g0) == set(g1)
    # the scorer's outputs are bit-identical, so what differs is the run-to-run noise of the fp32 atomics downstream;
    # the MLP Linear biases (true gradient zero in front of a train-mode BatchNorm) are nothing but that noise
    floor = grad_floor({k: v.cpu().numpy() for k, v in g0.items()})
    for k in g0:
        assert_close(g1[k], g0[k], 1e-4 if floor(k) > 0 else 1e-5, "grad " + k, floor=floor(k))
    for k in b0:
        assert_close(b1[k], b0[k], 1e-6, "buffer " + k)
