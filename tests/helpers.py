"""Shared test helpers: golden-fixture loading, tolerance checks and the CPU stand-in's installation."""
import glob
import json
import os
import re

import numpy as np
import torch

import emul_ops
from graph_neural_mapping_b200 import engine
from graph_neural_mapping_b200.models import discriminator as dmod
from graph_neural_mapping_b200.models import graphcnn as gmod
from graph_neural_mapping_b200.models import mlp as mlpmod
from graph_neural_mapping_b200.synth import SynthGraph

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# `seed0` of each case in tests/golden/make_golden.py: the numpy seed of its training step is 4242 + seed0
SEED0 = {"tiny_eps_sum": 100, "tiny_noeps_sum": 100, "tiny_eps_avg": 300, "tiny_noeps_avg": 300, "tiny_mlp1": 500,
         "tiny_mlp3": 500, "mid_eps_sum_h64": 900, "schaefer400_noeps": 0, "schaefer400_eps": 10, "tiny_eps_max": 700,
         "tiny_noeps_max": 700, "schaefer400_b16_noeps": 2000, "schaefer400_b16_eps": 2100}


def golden_names():
    return sorted(os.path.splitext(os.path.basename(p))[0] for p in glob.glob(os.path.join(GOLDEN_DIR, "*.npz")))


class Golden(object):
    def __init__(self, name):
        self.name = name
        self.z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
        self.cfg = json.loads(str(self.z["config"]))
        self.node_counts = self.z["node_counts"].tolist()
        self.labels = self.z["labels"].tolist()
        self.perm = self.z["perm"]

    def graphs(self):
        out = []
        if "edge_bits" in self.z.files:
            # compact fixtures: adjacency bitmaps; the edge order is synth.make_graph's canonical one
            # (upper-triangle pairs row-major, then the same pairs reversed, util.py:99-103)
            n = self.node_counts[0]
            bits = np.unpackbits(self.z["edge_bits"], axis=1)[:, :n * n].reshape(-1, n, n).astype(bool)
            for i in range(bits.shape[0]):
                iu, ju = np.nonzero(bits[i])
                em = torch.from_numpy(np.stack([np.concatenate([iu, ju]), np.concatenate([ju, iu])], 0).astype(np.int64))
                out.append(SynthGraph(n, self.labels[i], em, torch.eye(n, dtype=torch.float32)))
            return out
        eo = self.z["edge_off"]
        ec = self.z["edge_cat"]
        need_nb = self.cfg["neighbor_pooling_type"] == "max"
        for i, n in enumerate(self.node_counts):
            em = torch.from_numpy(ec[:, eo[i]:eo[i + 1]].copy())
            out.append(SynthGraph(n, self.labels[i], em, torch.eye(n, dtype=torch.float32), with_neighbors=need_nb))
        return out

    def state_dict(self):
        return {k[len("state/"):]: torch.from_numpy(self.z[k].copy()) for k in self.z.files if k.startswith("state/")}

    def group(self, prefix):
        return {k[len(prefix):]: self.z[k] for k in self.z.files if k.startswith(prefix)}

    def state_after_train(self):
        sd = self.state_dict()
        for k, v in self.group("buf_after/").items():
            sd[k] = torch.from_numpy(v.copy())
        return sd


def use_cpu_stand_in(monkeypatch):
    """Route every kernel call of the model code to the CPU stand-in (tests/emul_ops.py) for the current test."""
    for mod in (engine, gmod, mlpmod, dmod):
        monkeypatch.setattr(mod, "_ops", emul_ops)
    monkeypatch.setattr(engine, "require_cuda", lambda dev: None)


def build_model(g, sd=None):
    """The golden fixture's model on the CPU, with its initial state or `sd`."""
    c = g.cfg
    m = gmod.GIN_InfoMaxReg(c["num_layers"], c["num_mlp_layers"], c["input_dim"], c["hidden_dim"], c["output_dim"],
                            c["final_dropout"], c["learn_eps"], c["graph_pooling_type"], c["neighbor_pooling_type"],
                            torch.device("cpu"))
    m.load_state_dict(sd if sd is not None else g.state_dict())
    return m


def rel_err(a, b):
    """max|a-b| / max(|b|max, tiny): error relative to the tensor's scale (SURVEY 8(c))."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    scale = max(float(np.max(np.abs(b))) if b.size else 0.0, 1e-30)
    return float(np.max(np.abs(a - b))) / scale if b.size else 0.0


def assert_close(a, b, tol, what="", floor=0.0):
    a = np.asarray(a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a, dtype=np.float64)
    b = np.asarray(b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else b, dtype=np.float64)
    assert a.shape == b.shape, "%s: shape %s vs %s" % (what, a.shape, b.shape)
    nan_a, nan_b = np.isnan(a), np.isnan(b)
    assert (nan_a == nan_b).all(), "%s: NaN pattern differs" % what
    a = np.where(nan_a, 0.0, a)
    b = np.where(nan_b, 0.0, b)
    scale = max(float(np.max(np.abs(b))) if b.size else 0.0, floor, 1e-30)
    err = float(np.max(np.abs(a - b))) / scale if b.size else 0.0
    assert err <= tol, "%s: scaled error %.3e > %.1e" % (what, err, tol)
    return err


ZERO_GRAD_BIAS = re.compile(r"^mlps\.\d+\.(linear|linears\.\d+)\.bias$")


def grad_floor(grads, frac=1e-2, training=True):
    """Per-tensor comparison scale for gradients: returns f(name) -> floor for assert_close.

    Every gradient tensor is compared on ITS OWN max-abs scale (floor 0), so a regression in a small-gradient tensor
    (DGI bilinear weights, head biases, BatchNorm gamma/beta, eps) cannot hide behind the model's largest gradient.
    The one exception: a Linear bias inside an MLP always feeds a train-mode BatchNorm (mlp.py:48, graphcnn.py:163),
    so its true gradient is exactly zero and the reference's value is pure rounding noise (1e-16 .. 1e-20 of the
    others); those tensors are compared on a floor of `frac` x the model's largest gradient entry, i.e. they must be
    noise-small, not equal to the reference's noise. In eval mode (saliency parameter gradients) nothing is floored."""
    m = 0.0
    for v in grads.values():
        if v is not None and np.size(v):
            m = max(m, float(np.max(np.abs(np.asarray(v, dtype=np.float64)))))

    def floor_of(name):
        return frac * m if (training and ZERO_GRAD_BIAS.match(name)) else 0.0
    return floor_of
