"""GPU parity of the whole drop-in path (GIN_InfoMaxReg on libgnm) against the golden fixtures
written by the UNMODIFIED reference, and against the fp64 oracle (tolerance tie-breaker).

Tolerances, every tensor scaled by ITS OWN max-abs (SURVEY 8(c)): logits / loss / latent / BatchNorm buffers 1e-4;
every gradient tensor and saliency 3e-3 against the fp64 oracle, and 3e-3 plus the reference's own distance from that
oracle against the reference fixture. The gradient figure is set by ONE cancellation-limited tensor class at N = 400:
`mlps.3.linears.1.weight` of schaefer400_b16_eps, whose largest entry is 0.4 % of the model's largest gradient, is
1.1e-3 off the fp64 oracle in the reference's own fp32 run and 2.1e-3 off on the CUDA path (both sum 6400 cancelling
products in fp32, in different orders); every other tensor of every fixture is within 1e-3, most within 1e-5. Only the MLP Linear biases (true gradient exactly zero in front of a train-mode
BatchNorm) are compared on a floor (helpers.grad_floor). The `schaefer400_b16_*` fixtures have M = 6400 rows >= 4096:
they run the tcgen05 GEMM / aggregation kernels the benchmark runs, which the test asserts from libgnm's launch counters."""
import numpy as np
import pytest
import torch

from helpers import Golden, SEED0, assert_close, golden_names, grad_floor, rel_err
from oracle import gin_oracle
from graph_neural_mapping_b200.models import GIN_InfoMaxReg, Discriminator, MLP
from graph_neural_mapping_b200 import ops, synth

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda")
NAMES = golden_names()
TOL, TOL_GRAD = 1e-4, 3e-3
SEEDS = SEED0


def build_model(g, sd=None):
    c = g.cfg
    m = GIN_InfoMaxReg(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                       c["final_dropout"], c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"], DEV)
    m.load_state_dict(sd if sd is not None else g.state_dict())
    return m.to(DEV)


def train_step(model, graphs, beta, seed):
    model.train()
    np.random.seed(seed)
    c_logit, d_logit = model(graphs)
    labels = torch.LongTensor([x.label for x in graphs]).to(DEV)
    n = len(graphs) * graphs[0].node_features.shape[1]
    d_labels = torch.cat([torch.ones(n, 1), torch.zeros(n, 1)], 0).to(DEV)          # main.py:32
    loss = torch.nn.functional.cross_entropy(c_logit, labels) + beta * \
        torch.nn.functional.binary_cross_entropy_with_logits(d_logit, d_labels)     # main.py:34-37
    model.zero_grad()
    loss.backward()
    return c_logit, d_logit, loss


@pytest.mark.parametrize("name", NAMES)
def test_train_step_vs_reference_and_oracle(name):
    g = Golden(name)
    model = build_model(g)
    graphs = g.graphs()
    before = ops.launch_counts()
    c_logit, d_logit, loss = train_step(model, graphs, g.cfg["beta"], 4242 + SEEDS[name])
    ran = {k: v - before[k] for k, v in ops.launch_counts().items()}
    if "_b16_" in name:
        # the benchmarked code path: tcgen05 aggregation, tcgen05 Linear forward, tcgen05 dX and dW backward - and
        # none of the small-problem fallbacks
        assert ran["aggregate_tc"] >= 9 and ran["linear_tc"] >= 9, ran
        # (one-pass dX + dW kernel for the nine units with an input gradient, the dW kernel alone for the first)
        assert ran["linear_bwd_onepass_tc"] >= 8 and ran["linear_wgrad_tc"] + ran["linear_bwd_onepass_tc"] >= 9, ran
        assert ran["linear_ffma"] == ran["linear_bwd_ffma"] == ran["aggregate_csr"] == ran["aggregate_mma_sync"] == 0, ran
        assert not ops.aggregate_tc_status(), "a tcgen05 kernel hit its bounded wait"
    assert_close(c_logit, g.z["train/c_logit"], TOL, "c_logit")
    assert_close(d_logit, g.z["train/d_logit"], TOL, "d_logit")
    assert_close(loss, g.z["train/loss"], TOL, "loss")
    for k, v in g.group("buf_after/").items():
        got = model.state_dict()[k]
        if "num_batches" in k:
            assert int(got) == int(v)
        else:
            assert_close(got, v, TOL, k)
    # the fp64 oracle is the truth: every gradient tensor within TOL_GRAD of it on its own scale
    c = g.cfg
    ocfg = gin_oracle.OracleConfig(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                                   c["final_dropout"], c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"])
    r = gin_oracle.train_step_grads(g.state_dict(), graphs, g.perm, ocfg, c["beta"], torch.float64)
    assert_close(c_logit, r["c_logit"], TOL, "c_logit vs fp64")
    assert_close(d_logit, r["d_logit"], TOL, "d_logit vs fp64")
    ograds = {k: (v.numpy() if v is not None else None) for k, v in r["grads"].items()}
    floor = grad_floor(ograds)
    for k, p in model.named_parameters():
        if ograds.get(k) is not None:
            assert_close(p.grad, ograds[k], TOL_GRAD, "grad vs fp64 " + k, floor=floor(k))
    # the reference's own fp32 gradients carry summation-order noise of up to 1.1e-3 of a tensor's max-abs at N = 400
    # (measured here against the oracle, per tensor): the CUDA path must lie within TOL_GRAD plus that distance
    ref_grads = g.group("grad/")
    floor = grad_floor(ref_grads)
    for k, p in model.named_parameters():
        if k in ref_grads:
            assert p.grad is not None, k
            own = rel_err(ref_grads[k], ograds[k]) if floor(k) == 0.0 else 0.0
            assert own <= TOL_GRAD, "the reference itself is %.2e from the oracle on %s" % (own, k)
            assert_close(p.grad, ref_grads[k], TOL_GRAD + own, "grad " + k, floor=floor(k))
        else:
            assert p.grad is None, k


@pytest.mark.parametrize("name", NAMES)
def test_eval_latent_saliency_vs_reference(name):
    g = Golden(name)
    model = build_model(g, g.state_after_train())
    graphs = g.graphs()
    model.eval()
    np.random.seed(777)
    c_e, d_e = model(graphs)
    assert c_e.is_cuda and d_e.is_cuda and tuple(d_e.shape) == (2 * sum(g.node_counts), 1)
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
    if g.cfg["neighbor_pooling_type"] == "max":
        return      # the dummy row of max pooling is the batch-wide minimum (graphcnn.py:140): isolated nodes couple graphs
    # batched saliency == per-graph saliency (eval-mode BN, block-diagonal adjacency)
    cls = 1
    sb = model.compute_saliency_batched(graphs[:2], cls)
    n0 = g.node_counts[0]
    s0 = model.compute_saliency([graphs[0]], cls)
    s1 = model.compute_saliency([graphs[1]], cls)
    assert_close(sb[:n0], s0, 1e-6, "batched saliency g0")
    assert_close(sb[n0:], s1, 1e-6, "batched saliency g1")
    assert_close(s0, g.z["saliency/g0_c1"], TOL_GRAD, "saliency g0 vs reference")


def test_dropout_training_uses_torch_rng_and_keeps_shapes():
    g = Golden("tiny_eps_sum")
    c = g.cfg
    m = GIN_InfoMaxReg(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], 2, 0.5, True, "sum", "sum", DEV).to(DEV)
    m.train()
    graphs = g.graphs()
    torch.manual_seed(0)
    a, _ = m(graphs)
    torch.manual_seed(0)
    b, _ = m(graphs)
    # same torch seed -> same dropout mask (exact zeros coincide); the BatchNorm statistics are merged with
    # atomics (fp32 within a CTA, fp64 across CTAs), so the surviving values agree to rounding, not bitwise
    assert torch.equal(a == 0, b == 0) and bool((a == 0).any()) and tuple(a.shape) == (len(graphs), 2)
    assert torch.allclose(a, b, rtol=1e-3, atol=1e-4)


def test_adam_training_follows_reference_for_a_few_steps():
    """Three full main.py:25-41 steps (forward, loss, backward, Adam) against the fp32 oracle stepping the
    same state with torch.optim.Adam: parameters stay within tolerance (errors do not compound visibly)."""
    g = Golden("mid_eps_sum_h64")
    c = g.cfg
    model = build_model(g)
    graphs = g.graphs()
    opt = torch.optim.Adam(model.parameters(), lr=0.005)
    ocfg = gin_oracle.OracleConfig(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                                   0.0, c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"])
    sd = {k: v.clone() for k, v in g.state_dict().items()}
    names = [k for k, _ in model.named_parameters()]
    oparams = [sd[k].clone().double().requires_grad_(True) for k in names]
    oopt = torch.optim.Adam(oparams, lr=0.005)
    for step in range(3):
        np.random.seed(100 + step)
        perm = np.random.permutation(len(graphs))
        _, _, loss = train_step(model, graphs, c["beta"], 100 + step)
        opt.step()
        state = dict(sd)
        for k, p in zip(names, oparams):
            state[k] = p.detach()
        r = gin_oracle.train_step_grads(state, graphs, perm, ocfg, c["beta"], torch.float64)
        assert_close(loss, r["loss"], 5e-4, "loss step %d" % step)
        oopt.zero_grad()
        for k, p in zip(names, oparams):
            p.grad = r["grads"][k]
        oopt.step()
        for k, v in r["new_buffers"].items():
            sd[k] = v
    for k, p in zip(names, oparams):
        if k.startswith("mlps.") and k.endswith(".bias"):
            # a Linear bias feeding a train-mode BatchNorm has an exactly-zero true gradient; Adam turns its
            # rounding noise into +-lr steps (in the reference as well), and BatchNorm cancels the bias anyway
            continue
        assert_close(dict(model.named_parameters())[k], p.detach(), 5e-3, "param after 3 steps " + k)


def test_standalone_modules_on_gpu():
    torch.manual_seed(0)
    mlp = MLP(2, 20, 16, 16).to(DEV)
    x = torch.randn(300, 20, device=DEV, requires_grad=True)
    y = mlp(x)
    z = torch.nn.functional.batch_norm(x @ mlp.linears[0].weight.t() + mlp.linears[0].bias, None, None,
                                       mlp.batch_norms[0].weight, mlp.batch_norms[0].bias, True)
    yr = torch.relu(z) @ mlp.linears[1].weight.t() + mlp.linears[1].bias
    assert_close(y, yr, 2e-5, "mlp fwd")
    gy = torch.randn_like(y)
    ps = [x, mlp.linears[0].weight, mlp.linears[1].weight, mlp.batch_norms[0].weight, mlp.batch_norms[0].bias, mlp.linears[1].bias]
    g1 = torch.autograd.grad(y, ps, gy, retain_graph=True)
    g2 = torch.autograd.grad(yr, ps, gy)
    for a, b in zip(g1, g2):
        assert_close(a, b, 2e-4, "mlp grads")
    d = Discriminator(40).to(DEV)
    c = torch.rand(5, 40, device=DEV)
    hp, hm = torch.randn(60, 40, device=DEV, requires_grad=True), torch.randn(60, 40, device=DEV)
    out = d(c, hp, hm)
    cx = c.repeat_interleave(12, 0)
    ref = torch.cat([torch.nn.functional.bilinear(hp, cx, d.f_k.weight, d.f_k.bias),
                     torch.nn.functional.bilinear(hm, cx, d.f_k.weight, d.f_k.bias)], 0)
    assert_close(out, ref, 2e-5, "disc fwd")
    go = torch.randn_like(out)
    g1 = torch.autograd.grad(out, [hp, d.f_k.weight, d.f_k.bias], go, retain_graph=True)
    g2 = torch.autograd.grad(ref, [hp, d.f_k.weight, d.f_k.bias], go)
    for a, b in zip(g1, g2):
        assert_close(a, b, 2e-4, "disc grads")


def test_full_size_properties():
    """Size-independent checks at the benchmark's shape class (N=400, F=64, L=5; B=64 graphs here):
    aggregation of ones gives the degrees, eval forward is order-equivariant, saliency batching is exact."""
    torch.manual_seed(0)
    graphs = synth.make_graphs_bulk(64, 400, 30, 128, seed0=3, device="cuda")
    m = GIN_InfoMaxReg(5, 2, 400, 64, 2, 0.0, False, "sum", "sum", DEV).to(DEV).eval()
    np.random.seed(0)
    c, d = m(graphs)
    assert torch.isfinite(c).all() and torch.isfinite(d).all()
    bs = m._structure(graphs)
    rp, ci = bs.rowptr.cpu().numpy(), bs.colidx.cpu().numpy()
    assert rp[0] == 0 and rp[-1] == ci.size == 64 * (47600 + 400)
    rows = np.repeat(np.arange(rp.size - 1), np.diff(rp))
    assert np.all(ci // 400 == rows // 400)                                  # block diagonal
    key = rows.astype(np.int64) * (64 * 400) + ci
    assert np.all(np.diff(key) > 0)                                          # row-major sorted, no duplicates
    np.random.seed(0)
    c2, _ = m(list(reversed(graphs)))
    assert_close(c2.flip(0), c, 1e-5, "order equivariance")
    s_all = m.compute_saliency_batched(graphs[:3], 1)
    s_one = m.compute_saliency([graphs[1]], 1)
    assert_close(s_all[400:800], s_one, 1e-6, "batched saliency exact")


def test_cuda_graph_steps_match_eager_steps():
    """The captured forward/backward graphs (graphed.py) must reproduce the eager kernel-by-kernel path:
    same losses, gradients and BatchNorm buffers over several optimiser steps, with a different batch order
    and DGI permutation every step (those are the graphs' dynamic inputs)."""
    g = Golden("mid_eps_sum_h64")
    graphs = g.graphs()
    m_eager, m_graph = build_model(g), build_model(g)
    m_eager.use_cuda_graphs, m_graph.use_cuda_graphs = False, True
    # Linear biases that feed a train-mode BatchNorm have an exactly-zero true gradient; Adam would turn their
    # rounding noise into +-lr random walks that show up in running_mean. Keep them out of the optimiser here.
    def trainable(m):
        return [p for k, p in m.named_parameters() if not (k.startswith("mlps.") and k.endswith(".bias"))]
    o1 = torch.optim.Adam(trainable(m_eager), lr=0.005)
    o2 = torch.optim.Adam(trainable(m_graph), lr=0.005)
    rng = np.random.default_rng(0)
    for step in range(5):
        order = rng.permutation(len(graphs))
        batch = [graphs[i] for i in order]
        _, _, l1 = train_step(m_eager, batch, g.cfg["beta"], 50 + step)
        _, _, l2 = train_step(m_graph, batch, g.cfg["beta"], 50 + step)
        # the two arms differ by the arrival order of fp32 / fp64 atomics (BatchNorm sums, split-k partial products)
        assert_close(l2, l1.detach(), 5e-5, "loss step %d" % step)
        floor = grad_floor({k: p.grad.cpu().numpy() for k, p in m_eager.named_parameters() if p.grad is not None})
        for (k, p1), (_, p2) in zip(m_eager.named_parameters(), m_graph.named_parameters()):
            if p1.grad is None:
                assert p2.grad is None
            else:
                assert_close(p2.grad, p1.grad, 1e-4, "grad %s step %d" % (k, step), floor=floor(k))
        o1.step()
        o2.step()
    assert len(m_graph._plans) == 1 and next(iter(m_graph._plans.values())).bwd_graph is not None
    for (k, b1), (_, b2) in zip(m_eager.named_buffers(), m_graph.named_buffers()):
        if b1.dtype.is_floating_point:
            assert_close(b2, b1, 1e-4, k)
        else:
            assert int(b1) == int(b2) == 5
    # a stale backward is refused instead of silently using overwritten activations
    m_graph.train()
    np.random.seed(1)
    c_old, _ = m_graph(graphs)
    np.random.seed(2)
    m_graph(graphs)
    with pytest.raises(RuntimeError):
        c_old.sum().backward()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_gpu_data_parallel_matches_reference(world):
    """Launches tests/run_dp_gpu.py under torchrun with `world` ranks when the box has that many GPUs (skipped
    otherwise): sharded steps (model API and driver.Trainer) against the single-process reference fixtures - the
    B = 16 fixtures shard over 2, 4 and 8 ranks - plus the peer-memory exchange protocol."""
    import os
    import subprocess
    import sys
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    here = os.path.dirname(os.path.abspath(__file__))
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                          "--master-addr", "127.0.0.1", "--master-port", str(29371 + world), os.path.join(here, "run_dp_gpu.py")],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=900)
    assert "DP_GPU_CHECK_PASSED" in res.stdout, res.stdout[-3000:]


def test_schaefer1000_hidden128_config_vs_oracle():
    """BASELINE configs[3] shape class (N=1000 nodes, hidden 128): takes the general kernels - mma.sync block
    aggregation (N > 416), 128-wide feature slabs, unfused backward, chunked table-gradient merge."""
    torch.manual_seed(3)
    graphs = synth.make_graphs(2, n_rois=1000, n_time=300, seed0=77)
    for learn_eps in (True, False):
        model = GIN_InfoMaxReg(2, 2, 1000, 128, 2, 0.0, learn_eps, "sum", "sum", DEV).to(DEV)
        with torch.no_grad():
            model.eps.copy_(torch.tensor([0.2, -0.1]))
            for lin in model.linears_prediction:
                lin.weight.mul_(0.01)
        sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
        np.random.seed(5)
        perm = np.random.permutation(2)
        c_logit, d_logit, loss = train_step(model, graphs, 0.05, 5)
        ocfg = gin_oracle.OracleConfig(2, 2, 1000, 128, 2, 0.0, learn_eps, "sum", "sum")
        r = gin_oracle.train_step_grads(sd, graphs, perm, ocfg, 0.05, torch.float64)
        assert_close(c_logit, r["c_logit"], TOL, "c_logit")
        assert_close(d_logit, r["d_logit"], TOL, "d_logit")
        assert_close(loss, r["loss"], TOL, "loss")
        ograds = {k: (v.numpy() if v is not None else None) for k, v in r["grads"].items()}
        floor = grad_floor(ograds)
        for k, p in model.named_parameters():
            if ograds.get(k) is not None:
                assert_close(p.grad, ograds[k], TOL_GRAD, "grad " + k, floor=floor(k))
        s = model.compute_saliency([graphs[0]], 0)
        sref, _ = gin_oracle.saliency({k: v.detach().cpu() for k, v in model.state_dict().items()}, [graphs[0]], 0, ocfg)
        assert_close(s, sref, TOL_GRAD, "saliency")


def _loop_steps(model, graphs, beta, lr, seeds):
    opt = torch.optim.Adam(model.parameters(), lr=lr)
    losses = []
    for sd in seeds:
        np.random.seed(sd)
        c_logit, d_logit = model(graphs)
        labels = torch.LongTensor([x.label for x in graphs]).to(DEV)
        n = len(graphs) * graphs[0].node_features.shape[1]
        d_labels = torch.cat([torch.ones(n, 1), torch.zeros(n, 1)], 0).to(DEV)
        loss = torch.nn.functional.cross_entropy(c_logit, labels) + beta * \
            torch.nn.functional.binary_cross_entropy_with_logits(d_logit, d_labels)
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(float(loss))
    return losses


@pytest.mark.parametrize("name", ["mid_eps_sum_h64", "tiny_noeps_avg", "tiny_eps_max"])
def test_whole_step_trainer_matches_the_reference_loop(name):
    """driver.Trainer (SURVEY 8(f) N2: the whole step as one CUDA graph, Adam capturable) against main.py's loop body
    over the same model: per-step losses and the parameters / BatchNorm buffers after six steps (two eager warm-up
    steps, capture, three replays). Dropout off so that both arms see the same arithmetic."""
    from graph_neural_mapping_b200.driver import Trainer
    g = Golden(name)
    graphs = g.graphs()
    seeds = [11, 12, 13, 14, 15, 16]
    models = []
    for _ in range(2):
        m = build_model(g)
        m.final_dropout = 0.0
        m.train()
        models.append(m)
    ref_losses = _loop_steps(models[0], graphs, g.cfg["beta"], 0.01, seeds)
    tr = Trainer(models[1], lr=0.01, beta=g.cfg["beta"])
    got = []
    for sd in seeds:
        np.random.seed(sd)
        got.append(float(tr.step(graphs)))
    assert_close(np.array(got), np.array(ref_losses), 1e-4, "per-step losses")
    sd0, sd1 = models[0].state_dict(), models[1].state_dict()
    for k in sd0:
        if "num_batches" in k:
            assert int(sd0[k]) == int(sd1[k]), k
        elif (k.startswith("mlps") and ".linear" in k and k.endswith("bias")) or k.endswith("running_mean"):
            # zero-gradient biases in front of a train-mode BatchNorm: Adam random-walks on rounding noise, and the
            # running means carry those biases
            continue
        else:
            # Adam turns rounding noise on near-zero gradient entries into +-lr steps: 6 steps x lr 0.01 of slack
            assert_close(sd1[k], sd0[k], 6e-3, "after 6 steps: " + k)


def test_whole_step_trainer_with_dropout_is_reproducible():
    """With dropout on, the captured step uses torch's CUDA-graph aware Philox stream: two trainers seeded alike see
    the same masks, so their loss curves agree (to the rounding noise of the fp32 atomics in the gradient kernels)."""
    from graph_neural_mapping_b200.driver import Trainer
    g = Golden("mid_eps_sum_h64")
    graphs = g.graphs()
    curves = []
    for _ in range(2):
        m = build_model(g)
        m.train()
        torch.manual_seed(99)
        tr = Trainer(m, lr=0.01, beta=g.cfg["beta"])
        losses = []
        for sd in range(6):
            np.random.seed(100 + sd)
            losses.append(float(tr.step(graphs)))
        assert np.isfinite(losses).all()
        curves.append(np.array(losses))
    assert_close(curves[1], curves[0], 1e-4, "loss curve, run to run")
    assert abs(curves[0][-1] - curves[0][0]) > 1e-6, "parameters move"


@pytest.mark.parametrize("name", ["schaefer400_b16_noeps", "schaefer400_b16_eps"])
def test_whole_step_trainer_on_the_benchmarked_kernels_vs_reference(name):
    """driver.Trainer at M = 6400 rows (tcgen05 kernel family, asserted) against the UNMODIFIED reference's fixture:
    loss and every parameter gradient of the first step; then the captured CUDA graph (steps 3..) must reproduce the
    eager steps' loss on the same batch / permutation when the parameters are put back."""
    from graph_neural_mapping_b200.driver import Trainer
    g = Golden(name)
    graphs = g.graphs()
    model = build_model(g)
    model.final_dropout = 0.0
    model.train()
    tr = Trainer(model, lr=0.005, beta=g.cfg["beta"])
    before = ops.launch_counts()
    np.random.seed(4242 + SEEDS[name])
    loss = float(tr.step(graphs))
    ran = {k: v - before[k] for k, v in ops.launch_counts().items()}
    assert ran["aggregate_tc"] >= 9 and ran["linear_tc"] >= 9 and ran["linear_bwd_onepass_tc"] >= 8, ran
    assert ran["linear_ffma"] == ran["linear_bwd_ffma"] == 0, ran
    assert_close(np.array(loss), g.z["train/loss"], TOL, "loss of the first Trainer step")
    c = g.cfg
    ocfg = gin_oracle.OracleConfig(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                                   0.0, c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"])
    orc = gin_oracle.train_step_grads(g.state_dict(), graphs, g.perm, ocfg, c["beta"], torch.float64)["grads"]
    ref = g.group("grad/")
    floor = grad_floor(ref)
    for k, p in model.named_parameters():
        if k in ref:
            o = orc[k].numpy()
            assert_close(p.grad, o, TOL_GRAD, "Trainer grad vs fp64 " + k, floor=floor(k))
            own = rel_err(ref[k], o) if floor(k) == 0.0 else 0.0       # the reference's own fp32 noise on this tensor
            assert_close(p.grad, ref[k], TOL_GRAD + own, "Trainer grad " + k, floor=floor(k))
    losses = []
    for _ in range(4):                       # eager, capture, replay, replay - each from the fixture's state
        model.load_state_dict(g.state_dict())
        np.random.seed(4242 + SEEDS[name])
        losses.append(float(tr.step(graphs)))
    assert_close(np.array(losses), np.full(4, float(g.z["train/loss"])), TOL, "captured step vs reference loss")
    tr.finish()                              # raises if a tcgen05 kernel timed out


def test_trainer_learning_rate_schedule_reaches_the_captured_step():
    """main.py:138,147 decays the learning rate with StepLR every epoch. The Trainer keeps lr in a device tensor, so a
    scheduler step after capture changes the size of the next update (Adam's first-order step is ~lr per entry)."""
    from graph_neural_mapping_b200.driver import Trainer
    g = Golden("mid_eps_sum_h64")
    graphs = g.graphs()
    model = build_model(g)
    model.final_dropout = 0.0
    model.train()
    tr = Trainer(model, lr=0.01, beta=g.cfg["beta"])
    sched = torch.optim.lr_scheduler.StepLR(tr.optimizer, step_size=1, gamma=0.1)
    w = model.mlps[1].linears[0].weight

    def update_size():
        w0 = w.detach().clone()
        np.random.seed(5)
        tr.step(graphs)
        return float((w.detach() - w0).abs().max())

    for _ in range(4):
        big = update_size()                  # step 4 runs from the captured graph
    assert len(tr._plans) == 1 and next(iter(tr._plans.values())).graph is not None
    sched.step()                             # lr 0.01 -> 0.001
    assert abs(tr.get_lr() - 0.001) < 1e-9
    small = update_size()
    assert small < 0.3 * big, (big, small)
    tr.set_lr(0.01)
    again = update_size()
    assert again > 3.0 * small, (small, again)


@pytest.mark.parametrize("path", ["trainer", "model"])
def test_captured_step_follows_a_replaced_batchnorm_buffer(path):
    """A captured step bakes in the addresses of the BatchNorm buffers it updates. After four steps (Trainer: eager,
    eager, capture, replay; model(graphs) with CUDA graphs: eager, capture, replay, replay) one running_mean is replaced
    by a clone, as load_state_dict(assign=True) would: the next step must update the new tensor and count itself in
    num_batches_tracked, and leave the tensor the model no longer holds alone."""
    from graph_neural_mapping_b200.driver import Trainer
    g = Golden("mid_eps_sum_h64")
    graphs = g.graphs()
    model = build_model(g)
    model.train()
    model.use_cuda_graphs = True
    tr = Trainer(model, lr=0.01, beta=g.cfg["beta"]) if path == "trainer" else None

    def step(seed):
        if tr is not None:
            np.random.seed(seed)
            tr.step(graphs)
        else:
            train_step(model, graphs, g.cfg["beta"], seed)

    for sd in range(4):
        step(20 + sd)
    plans = tr._plans if tr is not None else model._plans
    plan = next(iter(plans.values()))
    assert len(plans) == 1 and (plan.graph if tr is not None else plan.bwd_graph) is not None
    bn = model.batch_norms[0]
    old = bn.running_mean
    bn.running_mean = old.clone()
    new, old_before, new_before = bn.running_mean, old.clone(), bn.running_mean.clone()
    count = int(bn.num_batches_tracked)
    step(30)
    torch.cuda.synchronize()
    assert not torch.equal(new, new_before), "the step did not update the model's running_mean"
    assert torch.equal(old, old_before), "the step wrote the replaced running_mean"
    assert int(bn.num_batches_tracked) == count + 1


def test_graph_store_stays_within_its_byte_budget():
    """Callers that build fresh graph objects every step must not leak device memory: the store drops its contents
    when the budget is exceeded and the results do not change."""
    g = Golden("mid_eps_sum_h64")
    model = build_model(g)
    model.eval()
    graphs = g.graphs()
    np.random.seed(0)
    want, _ = model(graphs)
    store = model._graph_store()
    store.max_bytes = 3 * store.bytes // 2
    for _ in range(6):
        fresh = g.graphs()                   # new objects, same content
        np.random.seed(0)
        got, _ = model(fresh)
        assert torch.equal(got, want)
        assert store.bytes <= 2 * store.max_bytes
    assert store.evictions >= 2 and len(store) <= 2 * len(graphs)


@pytest.mark.parametrize("name", ["mid_eps_sum_h64", "tiny_noeps_avg", "schaefer400_b16_noeps"])
def test_trainer_on_libgnm_step_kernels_matches_trainer_on_torch_ops(name):
    """A/B of the two Trainer paths: heads / dropout-free CE / BCE / Adam on libgnm's own kernels with the backward called
    directly (fused=True, no torch autograd in the step) against torch's loss functions, autograd and
    torch.optim.Adam(capturable=True) around the same encoder kernels (fused=False): per-step losses and the state
    after six steps (eager, eager, capture, three replays)."""
    from graph_neural_mapping_b200.driver import Trainer
    g = Golden(name)
    graphs = g.graphs()
    runs = []
    for fused in (False, True):
        m = build_model(g)
        m.final_dropout = 0.0
        m.train()
        tr = Trainer(m, lr=0.005, beta=g.cfg["beta"], fused=fused)
        losses = []
        for sd in range(6):
            np.random.seed(300 + sd)
            losses.append(float(tr.step(graphs)))
        tr.finish()
        runs.append((m, tr, np.array(losses)))
    # step 1 starts from identical parameters: only the loss kernels differ. Later steps carry Adam's amplification of
    # rounding noise on near-zero gradient entries (+-lr steps of random sign in either arm)
    assert_close(runs[1][2][:1], runs[0][2][:1], 5e-6, "first-step loss, libgnm step kernels vs torch ops")
    assert_close(runs[1][2], runs[0][2], 5e-4, "per-step losses, libgnm step kernels vs torch ops")
    sd0, sd1 = runs[0][0].state_dict(), runs[1][0].state_dict()
    for k in sd0:
        if "num_batches" in k:
            assert int(sd0[k]) == int(sd1[k]) == 6, k
        elif (k.startswith("mlps") and ".linear" in k and k.endswith("bias")) or k.endswith("running_mean"):
            continue          # zero-gradient biases: Adam random-walks on rounding noise (see the test above)
        elif "running_var" in k:
            assert_close(sd1[k], sd0[k], 2e-2, "after 6 steps: " + k)
        elif sd0[k].is_floating_point() and sd0[k].numel() > 1:
            # Adam turns the rounding noise of near-zero gradient entries into +-lr steps of random sign in either arm
            # (up to 2 * lr * steps apart); everything with a real gradient signal must move together: the typical
            # entry differs by a small fraction of one lr step
            diff = (sd1[k].double() - sd0[k].double()).abs()
            assert float(diff.max()) <= 2 * 0.005 * 6 + 1e-6, k
            assert float(diff.mean()) < 0.1 * 0.005, "after 6 steps: %s mean |diff| %.2e" % (k, float(diff.mean()))
    # the flat moments are the optimizer's state: a checkpoint taken from trainer.optimizer holds them
    tr = runs[1][1]
    osd = tr.optimizer.state_dict()
    assert len(osd["state"]) == len(tr._adam["offsets"]) and float(tr._adam["step"][0]) == 6.0
    st0 = next(iter(tr.optimizer.state.values()))
    assert float(st0["step"]) == 6.0 and float(st0["exp_avg_sq"].abs().sum()) > 0.0


def test_device_synth_and_streamed_result_files(tmp_path):
    """SURVEY 8(f) N3 on the GPU: graphs generated on the device with their edge lists LEFT on the device are ingested
    without a host trip and give the same model outputs as their host copies; `save_results` streams the saliency maps
    into .npy files that equal main.py:60-82's one-graph-per-call loops."""
    from graph_neural_mapping_b200 import driver
    dev_graphs = synth.make_graphs_bulk(70, 48, 30, 96, seed0=5, device="cuda", edges_on_device=True)
    host_graphs = synth.make_graphs_bulk(70, 48, 30, 96, seed0=5, device="cuda", edges_on_device=False)
    assert dev_graphs[0].edge_mat.is_cuda and not host_graphs[0].edge_mat.is_cuda
    for a, b in zip(dev_graphs, host_graphs):
        assert torch.equal(a.edge_mat.cpu(), b.edge_mat)
        e, half = b.edge_mat, b.edge_mat.shape[1] // 2
        # dataset.py:93-101: the top 30 % of ALL N*N entries (the N diagonal ones included) -> 0.3 N^2 - N directed
        # edges, give or take the symmetric pair the percentile value itself belongs to
        assert abs(e.shape[1] - (int(0.3 * 48 * 48) - 48)) <= 2 and torch.equal(e[:, half:], e[:, :half].flip(0))
    torch.manual_seed(1)
    m1 = GIN_InfoMaxReg(3, 2, 48, 16, 2, 0.0, False, "sum", "sum", DEV).to(DEV).eval()
    m2 = GIN_InfoMaxReg(3, 2, 48, 16, 2, 0.0, False, "sum", "sum", DEV).to(DEV).eval()
    m2.load_state_dict(m1.state_dict())
    h2d0 = m1._graph_store().h2d_bytes
    np.random.seed(0)
    c1, d1 = m1(dev_graphs)
    assert m1._graph_store().h2d_bytes - h2d0 < 70 * 48 * 8 + 4096          # no edge list crossed PCIe
    np.random.seed(0)
    c2, d2 = m2(host_graphs)
    assert torch.equal(c1, c2) and torch.equal(d1, d2)
    synth.release_edges(dev_graphs)                                          # the store holds the CSR / bitmaps
    np.random.seed(0)
    c3, _ = m1(dev_graphs)
    assert torch.equal(c3, c1)
    m1.forget_graphs()
    with pytest.raises(RuntimeError):
        m1(dev_graphs)                                                       # released edge lists cannot be rebuilt
    # result files (main.py:170-172), streamed
    out = driver.save_results(m2, host_graphs, str(tmp_path / "res"), batch=16)
    lat = np.load(out + "/latent_space.npy")
    sal = {c: np.load(out + "/saliency_%s.npy" % n) for c, n in ((0, "female"), (1, "male"))}
    labels = np.load(out + "/labels.npy")
    assert lat.shape == (70, 48) and lat.dtype == np.float32 and labels.shape == (70, 1)
    assert sal[0].shape == sal[1].shape == (70, 48, 48) and sal[0].dtype == np.float32
    for gi in (0, 15, 16, 69):
        for cls in (0, 1):
            ref = m2.compute_saliency([host_graphs[gi]], cls)                # main.py:64
            assert_close(sal[cls][gi], ref, 1e-6, "streamed saliency g%d c%d" % (gi, cls))
        np.random.seed(3)
        assert_close(lat[gi:gi + 1], m2([host_graphs[gi]], latent=True), 1e-5, "latent g%d" % gi)     # main.py:75-76
    assert np.array_equal(labels[:, 0], np.array([g.label for g in host_graphs]))
