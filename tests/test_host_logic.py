"""Host-logic tests (CPU): the engine's orchestration - graph store, batch assembly, the
hand-derived backward, saliency, data-parallel exchanges - run over a CPU stand-in for the
kernels (tests/emul_ops.py, injected here only) and compared with the golden fixtures that the
unmodified reference produced. The CUDA kernels are covered by the `-m gpu` tests."""
import numpy as np
import pytest
import torch

from helpers import Golden, SEED0, assert_close, build_model, golden_names, grad_floor, use_cpu_stand_in
from graph_neural_mapping_b200 import engine
from graph_neural_mapping_b200.models import mlp as mlpmod
from graph_neural_mapping_b200.models import discriminator as dmod

NAMES = golden_names()
TOL = 1e-4
TOL_GRAD = 2e-3


@pytest.fixture(autouse=True)
def cpu_backend(monkeypatch):
    use_cpu_stand_in(monkeypatch)


def train_step(model, graphs, g, seed):
    model.train()
    np.random.seed(seed)
    c_logit, d_logit = model(graphs)
    labels = torch.LongTensor([x.label for x in graphs])
    n = len(graphs) * graphs[0].node_features.shape[1]
    d_labels = torch.cat([torch.ones(n, 1), torch.zeros(n, 1)], 0)
    loss = torch.nn.functional.cross_entropy(c_logit, labels) + g.cfg["beta"] * \
        torch.nn.functional.binary_cross_entropy_with_logits(d_logit, d_labels)
    model.zero_grad()
    loss.backward()
    return c_logit, d_logit, loss


@pytest.mark.parametrize("name", NAMES)
def test_state_dict_layout_matches_reference(name):
    g = Golden(name)
    m = build_model(g)
    sd, ref = m.state_dict(), g.state_dict()
    assert list(sd.keys()) == list(ref.keys())
    for k in sd:
        assert tuple(sd[k].shape) == tuple(ref[k].shape) and sd[k].dtype == ref[k].dtype, k


@pytest.mark.parametrize("name", NAMES)
def test_train_step_vs_reference(name):
    g = Golden(name)
    if g.cfg["N"] >= 400:
        pytest.skip("dense CPU stand-in is too slow at N=400; covered on the GPU")
    model = build_model(g)
    graphs = g.graphs()
    c_logit, d_logit, loss = train_step(model, graphs, g, 4242 + SEED0[name])
    assert_close(c_logit, g.z["train/c_logit"], TOL, "c_logit")
    assert_close(d_logit, g.z["train/d_logit"], TOL, "d_logit")
    assert_close(loss, g.z["train/loss"], TOL, "loss")
    ref_grads = g.group("grad/")
    floor = grad_floor(ref_grads)
    for k, p in model.named_parameters():
        if k in ref_grads:
            assert p.grad is not None, k
            assert_close(p.grad, ref_grads[k], TOL_GRAD, "grad " + k, floor=floor(k))
        else:
            assert p.grad is None, k
    for k, v in g.group("buf_after/").items():
        got = model.state_dict()[k]
        if "num_batches" in k:
            assert int(got) == int(v)
        else:
            assert_close(got, v, TOL, k)


@pytest.mark.parametrize("name", NAMES)
def test_eval_latent_saliency_vs_reference(name):
    g = Golden(name)
    if g.cfg["N"] >= 400:
        pytest.skip("dense CPU stand-in is too slow at N=400; covered on the GPU")
    model = build_model(g, g.state_after_train())
    graphs = g.graphs()
    model.eval()
    np.random.seed(777)
    c_e, d_e = model(graphs)
    assert_close(c_e, g.z["eval/c_logit"], TOL, "eval c_logit")
    assert_close(d_e, g.z["eval/d_logit"], TOL, "eval d_logit")
    np.random.seed(1)
    lat = model(graphs, latent=True)
    assert isinstance(lat, np.ndarray) and lat.dtype == np.float32
    assert_close(lat, g.z["eval/latent"], TOL, "latent")
    np.random.seed(778)
    c1, d1 = model([graphs[0]])
    assert_close(c1, g.z["eval1/c_logit"], TOL, "eval1 c")
    assert_close(d1, g.z["eval1/d_logit"], TOL, "eval1 d")
    for k, v in g.group("saliency/").items():
        gi, cls = int(k[1:k.index("_")]), int(k[-1])
        s = model.compute_saliency([graphs[gi]], cls)
        assert tuple(s.shape) == v.shape
        assert_close(s, v, TOL_GRAD, "saliency " + k)
        if gi == 0 and cls == 1:
            ref = g.group("saliency_paramgrad/")
            floor = grad_floor(ref, training=False)
            for kk, p in model.named_parameters():
                if kk in ref:
                    assert_close(p.grad, ref[kk], TOL_GRAD, "saliency param grad " + kk, floor=floor(kk))
                else:
                    assert p.grad is None, kk
    if g.cfg["neighbor_pooling_type"] == "max":
        return      # the dummy row of max pooling is the batch-wide minimum (graphcnn.py:140): isolated nodes couple graphs
    sb = model.compute_saliency_batched(graphs[:2], 1)
    n0 = g.node_counts[0]
    assert_close(sb[:n0], g.z["saliency/g0_c1"], TOL_GRAD, "batched saliency g0")
    assert_close(sb[n0:], g.z["saliency/g1_c1"], TOL_GRAD, "batched saliency g1")


def test_one_numpy_draw_per_forward():
    g = Golden("tiny_eps_sum")
    model = build_model(g).eval()
    graphs = g.graphs()
    np.random.seed(5)
    model(graphs)
    after = np.random.rand()
    np.random.seed(5)
    np.random.permutation(len(graphs))
    assert after == np.random.rand()
    np.random.seed(5)
    model.compute_saliency([graphs[0]], 0)          # no numpy draw (graphcnn.py:254-299)
    after = np.random.rand()
    np.random.seed(5)
    assert after == np.random.rand()


def test_dense_feature_path_matches_gather_path():
    """Non-one-hot node features take the dense layer-0 path; on one-hot input scaled by 1 they agree."""
    g = Golden("tiny_eps_sum")
    graphs = g.graphs()
    m1, m2 = build_model(g), build_model(g)
    for gr in graphs:
        gr.node_features = gr.node_features.clone()
    graphs2 = g.graphs()
    for gr in graphs2:
        gr.node_features = gr.node_features * 1.0 + 0.0
        gr.node_features[0, 0] = 1.0000001   # not exactly one-hot any more -> dense path
    c1, d1, _ = train_step(m1, graphs, g, 3)
    c2, d2, _ = train_step(m2, graphs2, g, 3)
    assert_close(c2, c1.detach(), 1e-5, "dense vs gather c_logit")
    assert_close(d2, d1.detach(), 1e-5, "dense vs gather d_logit")
    floor = grad_floor({k: p.grad.numpy() for k, p in m1.named_parameters() if p.grad is not None})
    for (k, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        assert_close(p2.grad, p1.grad, 1e-4, "dense vs gather grad " + k, floor=floor(k))


def test_graph_store_reuse_and_errors():
    g = Golden("tiny_noeps_sum")
    model = build_model(g).eval()
    graphs = g.graphs()
    np.random.seed(0)
    a, _ = model(graphs)
    n_before = len(model._store)
    np.random.seed(0)
    b, _ = model(list(reversed(graphs)))
    assert len(model._store) == n_before == len(graphs)
    assert_close(b.flip(0), a.detach(), 1e-6, "order")
    bad = g.graphs()[0]
    bad.edge_mat = bad.edge_mat.clone()
    bad.edge_mat[0, 0] = 10 ** 6
    with pytest.raises(IndexError):
        model([bad])
    with pytest.raises(AssertionError):
        model.compute_saliency(graphs[:2], 0)


def test_mlp_and_discriminator_standalone():
    torch.manual_seed(0)
    mlp = mlpmod.MLP(3, 6, 5, 4)
    ref = torch.nn.Sequential()
    x = torch.randn(37, 6, requires_grad=True)
    y = mlp(x)
    h = x
    for j in range(2):
        h = torch.relu(torch.nn.functional.batch_norm(h @ mlp.linears[j].weight.t() + mlp.linears[j].bias, None, None,
                                                       mlp.batch_norms[j].weight, mlp.batch_norms[j].bias, True))
    yr = h @ mlp.linears[2].weight.t() + mlp.linears[2].bias
    assert_close(y, yr, 1e-5, "mlp fwd")
    gy = torch.randn_like(y)
    gx, = torch.autograd.grad(y, x, gy, retain_graph=True)
    gxr, = torch.autograd.grad(yr, x, gy)
    assert_close(gx, gxr, 1e-4, "mlp dx")
    with pytest.raises(ValueError):
        mlpmod.MLP(0, 3, 3, 3)
    d = dmod.Discriminator(7)
    c = torch.rand(3, 7)
    hp, hm = torch.randn(12, 7, requires_grad=True), torch.randn(12, 7)
    out = d(c, hp, hm)
    cx = c.repeat_interleave(4, 0)
    refo = torch.cat([torch.nn.functional.bilinear(hp, cx, d.f_k.weight, d.f_k.bias),
                      torch.nn.functional.bilinear(hm, cx, d.f_k.weight, d.f_k.bias)], 0)
    assert_close(out, refo, 1e-5, "disc fwd")
    go = torch.randn_like(out)
    g1 = torch.autograd.grad(out, [hp, d.f_k.weight, d.f_k.bias], go, retain_graph=True)
    g2 = torch.autograd.grad(refo, [hp, d.f_k.weight, d.f_k.bias], go)
    for a, b in zip(g1, g2):
        assert_close(a, b, 1e-4, "disc grads")


def test_csr_and_dense_aggregation_paths_agree(monkeypatch):
    g = Golden("tiny_eps_avg")
    graphs = g.graphs()
    m1, m2 = build_model(g), build_model(g)
    c1, d1, _ = train_step(m1, graphs, g, 9)
    assert m1._structure(graphs).bitmap_addr is not None         # 30 % dense -> tensor-core path selected
    monkeypatch.setattr(engine, "FORCE_CSR_AGGREGATE", True)
    c2, d2, _ = train_step(m2, graphs, g, 9)
    assert_close(c2, c1.detach(), 1e-5, "c_logit")
    assert_close(d2, d1.detach(), 1e-5, "d_logit")
    monkeypatch.setattr(engine, "DENSE_MIN_DENSITY", 0.9)
    assert m2._structure(graphs).bitmap_addr is None             # sparse batches stay on the CSR kernel


def test_fused_and_unfused_backward_agree(monkeypatch):
    g = Golden("tiny_mlp3")
    graphs = g.graphs()
    m1, m2 = build_model(g), build_model(g)
    train_step(m1, graphs, g, 21)
    monkeypatch.setattr(engine, "FORCE_UNFUSED_BACKWARD", True)
    train_step(m2, graphs, g, 21)
    floor = grad_floor({k: p.grad.numpy() for k, p in m1.named_parameters() if p.grad is not None})
    for (k, p1), (_, p2) in zip(m1.named_parameters(), m2.named_parameters()):
        if p1.grad is not None:
            assert_close(p2.grad, p1.grad, 1e-4, "grad " + k, floor=floor(k))


def test_no_reference_cycle_keeps_activations_alive():
    """The saved activations of a call must be freed by reference counting as soon as the outputs die (a
    self-referential autograd node once kept ~0.7 GB per batched saliency call alive until the cyclic GC ran)."""
    import gc
    g = Golden("tiny_eps_sum")
    model = build_model(g)
    graphs = g.graphs()
    model.compute_saliency_batched(graphs, 1)
    gc.collect()
    gc.disable()
    try:
        model.compute_saliency_batched(graphs, 1)
        np.random.seed(0)
        model.train()
        c_logit, d_logit = model(graphs)
        (c_logit.sum() + d_logit.sum()).backward()
        del c_logit, d_logit
        leaked = [o for o in gc.get_objects() if type(o).__name__ in ("_Saved", "Runner", "GINFunctionBackward")]
        assert not leaked, [type(o).__name__ for o in leaked]
    finally:
        gc.enable()


def test_shared_tag_sequence_takes_the_period_sum_path():
    """util.py:106-116 gives every subject the same (arbitrary) injective tag sequence; the layer-0 table gradient is
    then a sum over graphs (rows_period_sum). A batch whose graphs carry DIFFERENT tag orders must fall back to the
    scatter, and both must agree with the dense layer-0 path (which does not look at tags at all)."""
    g = Golden("tiny_eps_sum")
    n = g.graphs()[0].node_features.shape[0]
    perm = torch.from_numpy(np.random.RandomState(5).permutation(n))

    def batch(per_graph_shift, dense):
        graphs = g.graphs()
        for i, gr in enumerate(graphs):
            p = torch.roll(perm, i if per_graph_shift else 0)
            f = torch.zeros_like(gr.node_features)
            f[torch.arange(n), p] = 1.0
            if dense:
                f[0, p[0]] = 1.0000001                       # not exactly one-hot -> dense layer-0 path
            gr.node_features = f
        return graphs

    grads = {}
    for shift in (False, True):
        for dense in (False, True):
            m = build_model(g)
            graphs = batch(shift, dense)
            if not dense:
                assert m._structure(graphs).same_tags == (not shift)
            train_step(m, graphs, g, 17)
            grads[(shift, dense)] = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
    for shift in (False, True):
        floor = grad_floor({k: v.numpy() for k, v in grads[(shift, True)].items()})
        for k, v in grads[(shift, True)].items():
            assert_close(grads[(shift, False)][k], v, 1e-4, "shift=%s grad %s" % (shift, k), floor=floor(k))


def test_batched_evaluation_equals_the_one_graph_loops(tmp_path):
    """driver.class_logits / latent_space / saliency_maps / save_results against main.py:49-82's one-graph-per-forward
    loops over the same model, and against the reference's own per-graph outputs in the fixture."""
    from graph_neural_mapping_b200 import driver
    g = Golden("tiny_eps_sum")
    model = build_model(g, g.state_after_train())
    graphs = g.graphs()
    model.eval()
    loop_c = torch.cat([model([x])[0].detach() for x in graphs], 0)
    loop_lat = np.concatenate([model([x], latent=True) for x in graphs], 0)
    loop_s1 = np.stack([model.compute_saliency([x], 1).detach().cpu().numpy() for x in graphs], 0)
    assert_close(driver.class_logits(model, graphs, batch=3), loop_c, 1e-6, "class logits")
    lat, labels = driver.latent_space(model, graphs, batch=3)
    assert lat.dtype == np.float32 and labels.shape == (len(graphs), 1)
    assert_close(lat, loop_lat, 1e-6, "latent space")
    assert [int(v) for v in labels[:, 0]] == [x.label for x in graphs]
    s1 = driver.saliency_maps(model, graphs, 1, batch=3)
    assert s1.shape == loop_s1.shape
    assert_close(s1, loop_s1, 1e-6, "saliency maps")
    assert_close(s1[0], g.z["saliency/g0_c1"], TOL_GRAD, "saliency of graph 0 vs the reference")
    out = driver.save_results(model, graphs, str(tmp_path / "res"), batch=2)
    import os
    assert sorted(os.listdir(out)) == ["labels.npy", "latent_space.npy", "saliency_female.npy", "saliency_male.npy"]
    assert_close(np.load(os.path.join(out, "saliency_male.npy")), loop_s1, 1e-6, "saved saliency")
    assert np.load(os.path.join(out, "latent_space.npy")).shape == loop_lat.shape


def test_padded_neighbour_lists_follow_the_reference_order():
    """graphcnn.py:55-81: neighbours in `graph.neighbors` order, -1 pads up to the batch's max degree, the node itself
    last when learn_eps is False; the same lists come out of `edge_mat` alone (util.py:86-103 builds both from one
    edge iteration) when a graph object carries no `neighbors`."""
    g = Golden("tiny_noeps_max")
    with_nb = g.graphs()
    without = g.graphs()
    for x in without:
        x.neighbors = []
    for learn_eps in (False, True):
        m = build_model(g)
        m.learn_eps = learn_eps
        p1, f1 = m._padded_neighbours(with_nb)
        p2, f2 = m._padded_neighbours(without)
        assert torch.equal(p1, p2) and torch.equal(f1, f2)
        max_deg = max(x.max_neighbor for x in with_nb)
        assert p1.shape == (sum(len(x.g) for x in with_nb), max_deg + (0 if learn_eps else 1))
        start = 0
        for x in with_nb:
            for j, nb in enumerate(x.neighbors):
                want = [v + start for v in nb] + [-1] * (max_deg - len(nb)) + ([] if learn_eps else [start + j])
                assert p1[start + j].tolist() == want
                assert int(f1[start + j]) == (want[0] if nb else -1)
            start += len(x.g)


@pytest.mark.parametrize("name", ["tiny_eps_sum", "tiny_mlp1", "tiny_mlp3"])
def test_flat_params_and_buffers_cover_the_module(name):
    """engine.flat_params / flat_buffers (used to validate captured CUDA graphs every step) name exactly the tensors of
    model.parameters() minus the prediction heads, and of model.buffers()."""
    g = Golden(name)
    m = build_model(g)
    heads = {p.data_ptr() for p in m.linears_prediction.parameters()}
    want = {p.data_ptr() for p in m.parameters()} - heads
    assert {p.data_ptr() for p in engine.flat_params(m)} == want
    assert {b.data_ptr() for b in engine.flat_buffers(m)} == {b.data_ptr() for b in m.buffers()}
    assert len(engine.flat_buffers(m)) == len(list(m.buffers()))
