"""BatchNorm + ReLU on load: the tcgen05 aggregation reading a layer's pre-BatchNorm z (with that layer's graph pooling
formed from the same loads), the DGI / gather kernels reading z with a scale | shift table, and the training step that
no longer materialises h - each against the same computation on a materialised h = bn_relu_readout(z)."""
import numpy as np
import pytest
import torch

from helpers import Golden, SEED0, assert_close, grad_floor
from graph_neural_mapping_b200 import engine, ops
from graph_neural_mapping_b200.models import GIN_InfoMaxReg

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _batch(counts, seed, p=0.3):
    """Random symmetric graphs with self loops as the tcgen05 kernel sees them: (bitmap addresses, node offsets, n_max)."""
    rng = np.random.default_rng(seed)
    ems = []
    for n in counts:
        a = np.triu(rng.random((n, n)) < p, 1)
        r, c = np.nonzero(a | a.T)
        ems.append(np.stack([r, c]).astype(np.int64))
    edges = torch.from_numpy(np.concatenate(ems, 1) if ems else np.zeros((2, 0), np.int64)).to(DEV)
    eo = torch.from_numpy(np.cumsum([0] + [e.shape[1] for e in ems]).astype(np.int64)).to(DEV)
    no = torch.from_numpy(np.cumsum([0] + list(counts)).astype(np.int32)).to(DEV)
    m = int(sum(counts))
    rpl, cil, _ = ops.csr_build(edges, eo, no, len(counts), max(counts), m, True, True)
    words = [n * ((n + 31) // 32) for n in counts]
    bo = torch.from_numpy(np.cumsum([0] + words).astype(np.int64)).to(DEV)
    bm, dup = ops.bitmap_build(rpl, cil, no, bo, len(counts), int(sum(words)))
    assert int(dup.sum()) == 0
    addr = torch.tensor([bm.data_ptr() + 4 * int(o) for o in np.cumsum([0] + words)[:-1]], dtype=torch.int64, device=DEV)
    return bm, addr, no, max(counts), m


def _bn(f, seed):
    g = torch.Generator().manual_seed(seed)
    scale = (torch.rand(f, generator=g) + 0.5).to(DEV)
    shift = torch.randn(f, generator=g).to(DEV)
    shift[::3] = shift[::3].abs() + 0.1            # shift > 0 columns: relu(0*scale + shift) != 0 in the padding
    return scale, shift


RAGGED = [1, 416, 37, 129, 400, 63, 255, 2, 300, 65, 191, 7, 411, 128, 0, 64]


@pytest.mark.parametrize("counts", [[400] * 1024, RAGGED, [5, 17]])
@pytest.mark.parametrize("avg_pool", [False, True])
def test_aggregation_on_load_matches_readout_then_aggregate(counts, avg_pool):
    _bm, addr, no, n_max, m = _batch(counts, seed=len(counts))
    b, f = len(counts), 64
    torch.manual_seed(len(counts))
    z = torch.randn(m, f, device=DEV) * 2
    scale, shift = _bn(f, len(counts))
    ps = (1.0 / torch.tensor(counts, dtype=torch.float32).clamp(min=1)).to(DEV) if avg_pool else None
    h = torch.empty(m, f, device=DEV)
    g_ref = torch.empty(b, f, device=DEV)
    ops.bn_relu_readout(z, scale, shift, h, no, b, ps, g_ref)
    ref = torch.full((m, f), float("nan"), device=DEV)
    ops.aggregate_dense(addr, no, None, b, n_max, h, None, ref, 0, None, None, impl=2)
    out = torch.full((m, f), float("nan"), device=DEV)
    g_f = torch.full((b, 3 * f), float("nan"), device=DEV)
    pooled = g_f[:, f:2 * f]
    assert ops.aggregate_dense(addr, no, None, b, n_max, z, None, out, 0, None, None, bn_scale=scale, bn_shift=shift,
                               pooled=pooled, pool_scale=ps) is True
    assert not ops.aggregate_tc_status()
    # the activated rows are formed with the readout's expression: the aggregation is bit-identical
    assert torch.equal(out, ref)
    # the pooled sums add the same values in another order
    assert_close(pooled, g_ref, 1e-6, "pooled")
    assert torch.isnan(g_f[:, :f]).all() and torch.isnan(g_f[:, 2 * f:]).all()
    # without pooling: the same rows, nothing else written
    out2 = torch.full((m, f), float("nan"), device=DEV)
    assert ops.aggregate_dense(addr, no, None, b, n_max, z, None, out2, 0, None, None, bn_scale=scale, bn_shift=shift)
    assert torch.equal(out2, ref)


@pytest.mark.parametrize("case", ["n417", "eps", "average", "f128", "mma_sync"])
def test_aggregation_on_load_declines(case):
    counts = [417, 30] if case == "n417" else [30, 40]
    _bm, addr, no, n_max, m = _batch(counts, seed=5)
    f = 128 if case == "f128" else 64
    z = torch.randn(m, f, device=DEV)
    scale, shift = _bn(f, 1)
    out = torch.empty(m, f, device=DEV)
    rowptr = torch.zeros(m + 1, dtype=torch.int32, device=DEV)
    before = ops.kernels_recorded()
    ok = ops.aggregate_dense(addr, no, rowptr, 2, n_max, z, None, out, 1 if case == "average" else 0,
                             torch.tensor([0.1], device=DEV) if case == "eps" else None, None,
                             impl=1 if case == "mma_sync" else None, bn_scale=scale, bn_shift=shift,
                             pooled=torch.empty(2, f, device=DEV))
    assert ok is False
    assert ops.kernels_recorded() == before


@pytest.mark.parametrize("L,counts", [(5, [400] * 64), (5, RAGGED), (3, [33, 8, 129]), (1, [5])])
def test_dgi_kernels_on_load_match_materialised_h(L, counts):
    b, m, f = len(counts), int(sum(counts)), 64
    g = torch.Generator().manual_seed(L * 100 + b)
    z = torch.randn(L, m, f, generator=g).to(DEV)
    bn_all = torch.randn(L, 4, f, generator=g).to(DEV)
    bn_all[:, 0] = bn_all[:, 0].abs() + 0.5
    bn_all[:, 1, ::3] = bn_all[:, 1, ::3].abs()
    h = torch.empty(L, m, f, device=DEV)
    no = torch.from_numpy(np.cumsum([0] + list(counts)).astype(np.int32)).to(DEV)
    for l in range(L):
        ops.bn_relu_readout(z[l], bn_all[l, 0], bn_all[l, 1], h[l], no, b, None, None)
    bn = bn_all[:, :2]
    u = (0.2 * torch.randn(b, L * f, generator=g)).to(DEV)
    bias = torch.tensor([0.3], device=DEV)
    perm = torch.randperm(b, generator=g).to(torch.int32).to(DEV)
    table0 = ops.gather_nf_rows(h, b)
    table1 = ops.gather_nf_rows(z, b, bn=bn)
    assert torch.equal(table0, table1)

    def run(src, bnt):
        out = torch.empty(2 * m, 1, device=DEV)
        ops.dgi_score_fwd(src, u, table0, perm, no, b, bias, out, bn=bnt)
        dd = torch.randn(2 * m, generator=torch.Generator().manual_seed(9)).to(DEV)
        du, s2 = torch.empty(b, L * f, device=DEV), torch.empty(b, device=DEV)
        db = torch.zeros(1, dtype=torch.float64, device=DEV)
        ops.dgi_score_bwd(src, dd, table0, perm, no, b, du, s2, db, bn=bnt)
        tr = [torch.empty(2 * m, 1, device=DEV), torch.empty(m, device=DEV), torch.empty(b, L * f, device=DEV),
              torch.empty(b, device=DEV), torch.zeros(1, dtype=torch.float64, device=DEV),
              torch.zeros(1, dtype=torch.float64, device=DEV)]
        assert ops.dgi_score_train(src, u, table0, perm, no, b, bias, 1e-3, 1e-3, *tr, bn=bnt)
        return [out, du, s2, db] + tr

    # bit-identical activations: every fp32 output is equal; d_bias and the loss are fp64 atomics across graphs, whose
    # order varies from run to run
    names = ["out", "du", "s2", "d_bias", "train out", "d_score", "train du", "train s2", "train d_bias", "loss"]
    for nm, a, c in zip(names, run(h, None), run(z, bn)):
        if a.dtype == torch.float64:
            assert_close(c, a, 1e-12, nm)
        else:
            assert torch.equal(a, c), nm


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


@pytest.mark.parametrize("name", ["schaefer400_b16_noeps", "schaefer400_b16_eps"])
def test_trainer_step_on_load_matches_materialising_step(name, monkeypatch):
    """One eager Trainer step from the fixture's state, with h formed on load and with every h materialised: loss,
    every gradient and the BatchNorm buffers, each tensor on its own max-abs."""
    from graph_neural_mapping_b200.driver import Trainer
    g = Golden(name)
    graphs = g.graphs()
    runs = []
    for on_load in (False, True):
        with monkeypatch.context() as mp:
            mp.setattr(engine, "BN_ON_LOAD", on_load)
            calls = {}
            _counting(mp, ["bn_relu_readout"], calls)
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
    L = g.cfg["num_layers"]
    assert c0.get("bn_relu_readout") == L, c0
    # without learn_eps only the last layer's readout is left; under learn_eps every h is materialised as before
    assert c1.get("bn_relu_readout") == (L if g.cfg["learn_eps"] else 1), c1
    assert_close(np.array(loss1), np.array(loss0), 1e-6, "loss")
    assert set(g0) == set(g1)
    floor = grad_floor({k: v.cpu().numpy() for k, v in g0.items()})
    for k in g0:
        assert_close(g1[k], g0[k], 1e-4 if floor(k) > 0 else 1e-5, "grad " + k, floor=floor(k))
    for k in b0:
        assert_close(b1[k], b0[k], 1e-6, "buffer " + k)
