"""Pins the CPU oracle (oracle/) against outputs of the UNMODIFIED reference
(fixtures written by tests/golden/make_golden.py). CPU only."""
import numpy as np
import pytest
import torch

from oracle import csr_oracle, gin_oracle
from helpers import Golden, SEED0, assert_close, golden_names, grad_floor

# fp32 reference vs fp64 oracle: summation-order noise only. Scaled (max-abs) error.
TOL64 = 1e-4
TOL32 = 1e-4
TOL_GRAD = 2e-3


def _cfg(g):
    c = g.cfg
    return gin_oracle.OracleConfig(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"],
                                   c["output_dim"], c["final_dropout"], c["learn_eps"],
                                   c["graph_pooling_type"], c["neighbor_pooling_type"])


@pytest.mark.parametrize("name", golden_names())
def test_csr_indices_match_reference(name):
    g = Golden(name)
    if "adj_crow" not in g.z.files:
        pytest.skip("max pooling builds no Adj_block")
    graphs = g.graphs()
    ems = [x.edge_mat.numpy() for x in graphs]
    coo, m = csr_oracle.block_diag_coo(ems, g.node_counts, g.cfg["learn_eps"])
    assert np.array_equal(coo, g.z["adj_coo_idx"])
    rp, ci, val = csr_oracle.coalesced_csr(ems, g.node_counts, g.cfg["learn_eps"])
    assert np.array_equal(rp, g.z["adj_crow"])
    assert np.array_equal(ci, g.z["adj_col"])
    assert np.array_equal(val, g.z["adj_val"])
    rp2, ci2 = csr_oracle.multiset_csr(ems, g.node_counts, g.cfg["learn_eps"])
    assert np.array_equal(rp2, rp) and np.array_equal(ci2, ci)      # duplicate-free input
    off, scale = csr_oracle.graph_pool_segments(g.node_counts, g.cfg["graph_pooling_type"])
    pidx = g.z["pool_idx"]
    rows = np.repeat(np.arange(len(g.node_counts)), g.node_counts)
    assert np.array_equal(pidx[0], rows) and np.array_equal(pidx[1], np.arange(off[-1]))
    assert np.allclose(g.z["pool_val"], scale[rows].astype(np.float32))


def test_duplicate_edges_sum():
    em = np.array([[0, 1, 0, 2, 0], [1, 0, 1, 0, 2]], dtype=np.int64)   # edge (0,1) listed twice
    rp, ci, val = csr_oracle.coalesced_csr([em], [3], True)
    a = torch.sparse_coo_tensor(torch.from_numpy(em), torch.ones(5), (3, 3)).coalesce().to_sparse_csr()
    assert np.array_equal(rp, a.crow_indices().numpy()) and np.array_equal(ci, a.col_indices().numpy())
    assert np.array_equal(val, a.values().numpy())
    rp2, ci2 = csr_oracle.multiset_csr([em], [3], True)
    assert rp2.tolist() == [0, 3, 4, 5] and ci2.tolist() == [1, 1, 2, 0, 0]
    assert np.array_equal(csr_oracle.dense_adjacency([em], [3], True), a.to_dense().numpy())


@pytest.mark.parametrize("name", golden_names())
@pytest.mark.parametrize("dtype,tol", [(torch.float64, TOL64), (torch.float32, TOL32)])
def test_train_step_matches_reference(name, dtype, tol):
    g = Golden(name)
    if dtype == torch.float32 and g.cfg["N"] >= 400:
        pytest.skip("fp32 dense oracle at N=400 adds nothing over fp64")
    r = gin_oracle.train_step_grads(g.state_dict(), g.graphs(), g.perm, _cfg(g), g.cfg["beta"], dtype)
    assert_close(r["c_logit"], g.z["train/c_logit"], tol, "c_logit")
    assert_close(r["d_logit"], g.z["train/d_logit"], tol, "d_logit")
    assert_close(r["loss"], g.z["train/loss"], tol, "loss")
    floor = grad_floor(g.group("grad/"))
    for k, v in g.group("grad/").items():
        assert_close(r["grads"][k], v, TOL_GRAD, "grad " + k, floor=floor(k))
    for k in g.group("gradnone/"):
        assert r["grads"][k] is None, k
    for k, v in g.group("buf_after/").items():
        if "num_batches" in k:
            assert int(r["new_buffers"][k]) == int(v)
        else:
            assert_close(r["new_buffers"][k], v, tol, k)


@pytest.mark.parametrize("name", golden_names())
def test_eval_and_saliency_match_reference(name):
    g = Golden(name)
    cfg = _cfg(g)
    sd = {k: (v.double() if v.is_floating_point() else v) for k, v in g.state_after_train().items()}
    graphs = g.graphs()
    with torch.no_grad():
        r = gin_oracle.forward(sd, graphs, g.z["eval/perm"], cfg, training=False)
    assert_close(r["c_logit"], g.z["eval/c_logit"], TOL64, "eval c_logit")
    assert_close(r["d_logit"], g.z["eval/d_logit"], TOL64, "eval d_logit")
    assert_close(r["g_f"], g.z["eval/latent"], TOL64, "latent")
    with torch.no_grad():
        r1 = gin_oracle.forward(sd, graphs[:1], np.array([0]), cfg, training=False)
    assert_close(r1["c_logit"], g.z["eval1/c_logit"], TOL64, "eval1 c_logit")
    assert_close(r1["d_logit"], g.z["eval1/d_logit"], TOL64, "eval1 d_logit")
    for k, v in g.group("saliency/").items():
        gi, cls = int(k[1:k.index("_")]), int(k[-1])
        s, _ = gin_oracle.saliency(sd, [graphs[gi]], cls, cfg)
        assert_close(s, v, TOL_GRAD, "saliency " + k)
    # batching saliency is exact in eval mode (SURVEY A10)
    # (not for max pooling: its dummy row is the batch-wide minimum, graphcnn.py:140)
    if len(graphs) >= 2 and "saliency/g1_c1" in g.z.files and g.cfg["neighbor_pooling_type"] != "max":
        s, _ = gin_oracle.saliency(sd, graphs[:2], 1, cfg)
        n0 = g.node_counts[0]
        assert_close(s[:n0], g.z["saliency/g0_c1"], TOL_GRAD, "batched saliency g0")
        assert_close(s[n0:], g.z["saliency/g1_c1"], TOL_GRAD, "batched saliency g1")


@pytest.fixture
def golden_threads():
    """The intra-op thread count tests/golden/make_golden.py ran the reference with. ATen splits its CPU reductions by
    thread count, so only with the same count does the port repeat the reference's summation order, whatever the host's
    core count."""
    saved = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(saved)


@pytest.mark.parametrize("name", [n for n in golden_names() if "max" not in n])
def test_aten_port_matches_reference(name, golden_threads):
    """oracle/aten_port.py (the CPU baseline that bench.py times) against the reference's outputs."""
    from oracle import aten_port
    g = Golden(name)
    sd = {}
    for k, v in g.state_dict().items():
        sd[k] = v.clone().requires_grad_(True) if (v.is_floating_point() and "running_" not in k) else v.clone()
    seed = 4242 + SEED0[name]
    np.random.seed(seed)
    graphs = g.graphs()
    c_logit, d_logit, g_f = aten_port.forward(sd, graphs, g.cfg, True)
    assert_close(c_logit, g.z["train/c_logit"], 1e-6, "c_logit")
    assert_close(d_logit, g.z["train/d_logit"], 1e-6, "d_logit")
    labels = torch.LongTensor(g.labels)
    n = len(graphs) * g.cfg["N"]
    d_labels = torch.cat([torch.ones(n, 1), torch.zeros(n, 1)], 0)
    loss = torch.nn.functional.cross_entropy(c_logit, labels) + g.cfg["beta"] * \
        torch.nn.functional.binary_cross_entropy_with_logits(d_logit, d_labels)
    loss.backward()
    floor = grad_floor(g.group("grad/"))
    for k, v in g.group("grad/").items():
        assert_close(sd[k].grad, v, 1e-5, "grad " + k, floor=floor(k))
