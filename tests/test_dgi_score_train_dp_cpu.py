"""Data-parallel host logic of the training step's one-pass DGI scorer on CPU: world_size 2 over gloo, kernels replaced by
the CPU stand-in (tests/emul_ops.py) plus a stand-in of gnm_dgi_score_train composed of the three calls it replaces.
On every rank, engine.run_forward(bce=...) + run_backward (scores, loss and the scorer's backward from the forward pass:
negatives broadcast from rank 0, s2 feeding the reduced negative-row gradients) must give the loss and the gradients of
the three-call path (run_forward, BCE on d_logit, run_backward)."""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _bce_terms(x, m, grad_scale):
    """BCEWithLogits against main.py:32's targets (first m scores 1, the rest 0): per-score loss and gradient."""
    y = torch.cat([torch.ones(m), torch.zeros(m)])
    loss = torch.clamp(x, min=0) - x * y + torch.log1p(torch.exp(-x.abs()))
    return loss, (torch.sigmoid(x) - y) * grad_scale


def _worker(rank, world, port, name, seed, out_dir):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import torch.distributed as td
    import emul_ops
    from helpers import Golden
    from graph_neural_mapping_b200 import dist as gdist, engine
    from graph_neural_mapping_b200.models import graphcnn as gmod, mlp as mlpmod, discriminator as dmod

    def dgi_score_train(h_all, u, neg_table, neg_idx, node_off, n_graphs, bias, grad_scale, loss_scale, out, d_score, du,
                        s2, d_bias, loss_acc):
        emul_ops.dgi_score_fwd(h_all, u, neg_table, neg_idx, node_off, n_graphs, bias, out)
        m = h_all.shape[1]
        terms, dd = _bce_terms(out.view(-1), m, grad_scale)
        loss_acc += loss_scale * terms.double().sum()
        d_score.copy_(dd[:m])
        emul_ops.dgi_score_bwd(h_all, dd, neg_table, neg_idx, node_off, n_graphs, du, s2, d_bias)
        return True

    torch.set_num_threads(1)
    emul_ops.dgi_score_train = dgi_score_train
    engine._ops = emul_ops
    mlpmod._ops = emul_ops
    dmod._ops = emul_ops
    engine.require_cuda = lambda dev: None
    td.init_process_group("gloo", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    comm = gdist.Comm(None, world, rank)
    g = Golden(name)
    c = g.cfg
    model = gmod.GIN_InfoMaxReg(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                                c["final_dropout"], c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"],
                                torch.device("cpu"))
    model.set_comm(comm)
    model.train()
    graphs = gdist.shard(g.graphs(), comm)
    np.random.seed(seed)
    neg_idx = torch.from_numpy(np.random.permutation(len(graphs) * world).astype(np.int32))
    out = {}
    for arm in ("three_calls", "one_pass"):
        model.load_state_dict(g.state_dict())
        bs = model._structure(graphs)
        params = [p.detach() for p in engine.flat_params(model)]
        m = bs.n_rows
        w = c["beta"] / (2.0 * m)
        loss = torch.zeros(1, dtype=torch.float64)
        if arm == "one_pass":
            _, _, sv = engine.run_forward(model, bs, neg_idx, True, True, None, params, comm, bce=(w, w, loss))
            assert sv.scored is not None
            dd = None
        else:
            _, d_logit, sv = engine.run_forward(model, bs, neg_idx, True, True, None, params, comm)
            assert sv.scored is None
            terms, dd = _bce_terms(d_logit.view(-1), m, w)
            loss += w * terms.double().sum()
            dd = dd.view(-1, 1)
        _, grads = engine.run_backward(model, sv, params, None, dd, False, comm)
        out[arm + "/loss"] = loss.numpy()
        names = {id(p): k for k, p in model.named_parameters()}
        for p, gr in zip(engine.flat_params(model), grads):
            k = names[id(p)]
            if gr is not None:
                out[arm + "/grad/" + k] = gr.reshape(-1).numpy()
    np.savez(os.path.join(out_dir, "rank%d.npz" % rank), **out)
    td.barrier()
    td.destroy_process_group()


@pytest.mark.parametrize("name,seed", [("mid_eps_sum_h64", 5142), ("tiny_noeps_sum", 4342)])
def test_two_ranks_one_pass_scorer_matches_three_calls(name, seed, tmp_path):
    sys.path.insert(0, HERE)
    from helpers import Golden, assert_close
    world = 2
    g = Golden(name)
    if g.cfg["B"] % world:
        pytest.skip("batch not divisible")
    port = _free_port()
    mp.spawn(_worker, args=(world, port, name, seed, str(tmp_path)), nprocs=world, join=True)
    for rank in range(world):
        r = np.load(os.path.join(str(tmp_path), "rank%d.npz" % rank))
        assert_close(r["one_pass/loss"], r["three_calls/loss"], 1e-12, "rank %d loss" % rank)
        keys = sorted(k[len("three_calls/"):] for k in r.files if k.startswith("three_calls/grad/"))
        assert keys == sorted(k[len("one_pass/"):] for k in r.files if k.startswith("one_pass/grad/"))
        assert "grad/disc.f_k.bias" in keys and "grad/disc.f_k.weight" in keys
        for k in keys:
            assert_close(r["one_pass/" + k], r["three_calls/" + k], 1e-6, "rank %d %s" % (rank, k))
