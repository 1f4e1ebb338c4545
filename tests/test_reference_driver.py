"""The reference's OWN driver (`main.py`, staged unmodified in oracle/_ref by oracle/make_ref.py) executed against the
repo-root `models/` shim - the drop-in claim of SURVEY 8(b): `from models.graphcnn import *` (main.py:9) resolves to
the libgnm-backed classes and `train()` / `test()` / `get_saliency_map()` / `get_latent_space()` (main.py:19-96) run
unchanged. The same functions run on the reference's own classes on the CPU give the expected values.

Why these tests skip in a plain checkout: both sides of the comparison execute the reference's own sources (main.py and
its models/), which this repository does not contain. `python oracle/make_ref.py` stages them, byte for byte, into the
git-ignored oracle/_ref from a checkout of the original project named by GNM_REFERENCE_ROOT; build() does the same when
that checkout is present. The expected values cannot be stored instead: they are main.py's outputs on the reference's
classes, so writing them needs those same sources. What the reference's classes compute on these graphs (train step,
eval logits, latent, saliency) is stored in tests/golden/ and checked there against this repository's models."""
import argparse
import warnings

import numpy as np
import pytest
import torch

from helpers import Golden, assert_close
from oracle import ref_arm

needs_ref = pytest.mark.skipif(not ref_arm.available(), reason="oracle/_ref not staged (python oracle/make_ref.py)")


def _args(batch_size, iters):
    return argparse.Namespace(batch_size=batch_size, iters_per_epoch=iters)


def _model(main_mod, g, device, final_dropout=0.0):
    c = g.cfg
    m = main_mod.GIN_InfoMaxReg(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                                final_dropout, c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"],
                                device).to(device)
    m.load_state_dict(g.state_dict())
    return m


def _drive(main_mod, g, device, graphs):
    """What main.py:143-172 does with a model, in miniature: evaluation loops, then one epoch of training."""
    out = {}
    model = _model(main_mod, g, device)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        np.random.seed(21)
        out["test"] = main_mod.test(None, model, device, graphs)                       # main.py:85-96
        np.random.seed(22)
        out["latent"], out["labels"] = main_mod.get_latent_space(model, graphs)        # main.py:71-82
        out["saliency0"] = main_mod.get_saliency_map(model, graphs[:2], 0)             # main.py:60-68
        out["saliency1"] = main_mod.get_saliency_map(model, graphs[:2], 1)
        np.random.seed(23)
        c, d = main_mod.pass_data_iteratively(model, graphs)                           # main.py:49-57
        out["c_logit"], out["d_logit"] = c.detach().cpu().numpy(), d.detach().cpu().numpy()
        model = _model(main_mod, g, device)
        opt = torch.optim.Adam(model.parameters(), lr=0.005)                            # main.py:136
        np.random.seed(24)
        out["train_loss"] = main_mod.train(_args(len(graphs) - 1, 3), model, device, graphs, opt, g.cfg["beta"], 0)
    return out


@needs_ref
def test_staged_reference_is_unmodified_and_runs():
    files = ref_arm.verify()
    assert "main.py" in files and "models/graphcnn.py" in files
    g = Golden("tiny_eps_sum")
    main_ref = ref_arm.reference_main("reference")
    assert main_ref.GIN_InfoMaxReg.__module__ == "models.graphcnn"
    out = _drive(main_ref, g, torch.device("cpu"), g.graphs())
    assert np.isfinite(out["train_loss"]) and out["latent"].shape == (g.cfg["B"], g.cfg["num_layers"] * g.cfg["hidden_dim"])
    # the fixture was written by the same classes: its eval latent is reproduced from the trained buffers' state
    cls = ref_arm.reference_model_class()
    assert cls.__module__ == "gnm_reference_graphcnn"


@needs_ref
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tiny_eps_sum", "tiny_noeps_avg", "mid_eps_sum_h64"])
def test_reference_main_runs_unchanged_on_the_repo_models(name):
    g = Golden(name)
    graphs = g.graphs()
    want = _drive(ref_arm.reference_main("reference"), g, torch.device("cpu"), graphs)
    main_repo = ref_arm.reference_main("repo")
    assert main_repo.GIN_InfoMaxReg.__module__.startswith("graph_neural_mapping_b200.")
    got = _drive(main_repo, g, torch.device("cuda"), graphs)
    assert got["test"] == want["test"], (got["test"], want["test"])                    # accuracy, precision, recall
    assert np.array_equal(got["labels"], want["labels"])
    assert got["latent"].dtype == want["latent"].dtype == np.float32
    assert_close(got["latent"], want["latent"], 1e-4, "get_latent_space")
    assert_close(got["c_logit"], want["c_logit"], 1e-4, "pass_data_iteratively c_logit")
    assert_close(got["d_logit"], want["d_logit"], 1e-4, "pass_data_iteratively d_logit")
    assert got["saliency0"].shape == want["saliency0"].shape
    assert_close(got["saliency0"], want["saliency0"], 2e-3, "get_saliency_map cls 0")
    assert_close(got["saliency1"], want["saliency1"], 2e-3, "get_saliency_map cls 1")
    # three Adam steps of main.py:25-43 on batches of B-1 graphs drawn by the driver's own np.random.permutation
    assert_close(np.array(got["train_loss"]), np.array(want["train_loss"]), 5e-4, "train() average loss")
