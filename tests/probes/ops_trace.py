"""Call trace of the kernel entry points the engine reaches; a refactor of the host orchestration must leave it as it is.

The ops module seen by engine, graphcnn, mlp, discriminator and driver is replaced by a shim that passes every attribute through
and records each call of a public function: its name, every argument bound to the callee's signature (defaults filled
in, so a positional and a keyword spelling of one call record alike) and any boolean return. A tensor is recorded as
shape, dtype, strides and storage offset (which places the views of engine._ZeroPool's buffers), None as None, a
scalar as its value, an ops.BnTail as its kind and count; no pointer value is recorded. Per case the probe prints one
digest of the trace and one of the case's outputs (parameter gradients, saliency maps, ROI averages) as raw bytes;
`--dump DIR` also writes each full trace, one call per line, to diff.

  cpu: the CPU stand-in kernels (tests/emul_ops.py). Every golden fixture with N < 400 through a training step,
       compute_saliency, compute_saliency_batched and compute_roi_saliency_batched((0, 1)); the same under
       FORCE_CSR_AGGREGATE and under FORCE_UNFUSED_BACKWARD; a batch whose node features are not exactly one-hot; and
       every such fixture through compute_integrated_gradients_batched with return_delta (a points_per_pass that splits
       a graph's points over two passes, and one that packs several graphs per pass) and compute_roi_occlusion_batched at
       two occlusions_per_pass that split differently. A call that raises ValueError records its message. Deterministic:
       both digests are compared bit for bit.
  gpu: the libgnm kernels. Trainer steps (fused and not: the two eager warm-up steps, the capture and a replay),
       model(graphs) + backward with CUDA graphs on (the eager first sighting, the capture and a replay), then with CUDA
       graphs off model(graphs) + backward at 1024 x 400, learn_eps, average pooling with an isolated node, max pooling,
       hidden width 128, ROI saliency (one-hot, dense, max pooling) and the integrated-gradients and occlusion calls of
       the cpu mode on the same models. A capture records its calls, a replay none. Only the trace digests are meant to
       match across builds: the kernels' float atomics make outputs differ in the last bits.

The launch counter readers (ops.launch_counts, kernels_recorded, kernels_launched) are not recorded: they launch
nothing, and which module reads them around a capture is plumbing.

    python tests/probes/ops_trace.py cpu|gpu [--dump DIR]"""
import argparse
import hashlib
import inspect
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from graph_neural_mapping_b200 import driver, engine, graphed, synth  # noqa: E402
from graph_neural_mapping_b200.models import GIN_InfoMaxReg  # noqa: E402
from graph_neural_mapping_b200.models import discriminator as dmod  # noqa: E402
from graph_neural_mapping_b200.models import graphcnn as gmod  # noqa: E402
from graph_neural_mapping_b200.models import mlp as mlpmod  # noqa: E402

USERS = (engine, gmod, mlpmod, dmod, driver, graphed)
COUNTERS = ("launch_counts", "kernels_recorded", "kernels_launched")


def _sig(v):
    if torch.is_tensor(v):
        return ("T", tuple(v.shape), str(v.dtype).replace("torch.", ""), tuple(v.stride()), v.storage_offset())
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    if isinstance(v, (list, tuple)):
        return tuple(_sig(x) for x in v)
    if isinstance(v, np.ndarray):
        return ("A", v.shape, str(v.dtype))
    if type(v).__name__ == "BnTail":
        return ("BnTail", int(v.struct.kind), float(v.struct.count))
    return type(v).__name__


class TracingOps(object):
    """Pass-through view of an ops module that records the calls of its public functions in `self.trace`."""

    def __init__(self, base):
        self._base = base
        self.trace = []

    def __getattr__(self, name):
        attr = getattr(self._base, name)
        if name.startswith("_") or name in COUNTERS or not inspect.isfunction(attr):
            return attr
        params = inspect.signature(attr)
        trace = self.trace

        def traced(*args, **kwargs):
            bound = params.bind(*args, **kwargs)
            bound.apply_defaults()
            ret = attr(*args, **kwargs)
            rec = (name, tuple((k, _sig(v)) for k, v in bound.arguments.items()))
            trace.append(rec + ((("ret", ret),) if isinstance(ret, bool) else ()))
            return ret
        return traced


class Case(object):
    def __init__(self, shim):
        self.shim = shim
        self.outputs = hashlib.sha256()

    def __enter__(self):
        del self.shim.trace[:]
        return self

    def __exit__(self, *exc):
        return False

    def add(self, t):
        if t is None:
            self.outputs.update(b"None")
            return
        t = t.detach().float().cpu().contiguous()
        self.outputs.update(str(tuple(t.shape)).encode())
        self.outputs.update(t.numpy().tobytes())

    def add_grads(self, model):
        for _, p in model.named_parameters():
            self.add(p.grad)


def _digest(trace):
    return hashlib.sha256("\n".join(repr(c) for c in trace).encode()).hexdigest()[:16]


def report(name, case, dump):
    trace = case.shim.trace
    print("%-44s calls %5d  trace %s  outputs %s" % (name, len(trace), _digest(trace), case.outputs.hexdigest()[:16]),
          flush=True)
    if dump:
        with open(os.path.join(dump, name + ".txt"), "w") as f:
            f.write("\n".join(repr(c) for c in trace) + "\n")


def _train_step(model, graphs, beta, seed):
    model.train()
    np.random.seed(seed)
    c_logit, d_logit = model(graphs)
    dev = c_logit.device
    labels = torch.tensor([g.label for g in graphs], device=dev)
    n = sum(len(g.g) for g in graphs)
    d_labels = torch.cat([torch.ones(n, 1), torch.zeros(n, 1)], 0).to(dev)
    loss = torch.nn.functional.cross_entropy(c_logit, labels) + beta * \
        torch.nn.functional.binary_cross_entropy_with_logits(d_logit, d_labels)
    model.zero_grad()
    loss.backward()
    return c_logit, d_logit


def run_model_cases(case, model, graphs, beta, seed, roi_per_graph=False):
    """A training step, compute_saliency of graph 0, compute_saliency_batched and the ROI averages, outputs hashed."""
    c_logit, d_logit = _train_step(model, graphs, beta, seed)
    case.add(c_logit)
    case.add(d_logit)
    case.add_grads(model)
    case.add(model.compute_saliency([graphs[0]], 1))
    case.add_grads(model)
    case.add(model.compute_saliency_batched(graphs[:2], 0))
    case.add_grads(model)
    if roi_per_graph:
        for g in graphs[:2]:
            case.add(model.compute_roi_saliency_batched([g], (0, 1)))
    else:
        case.add(model.compute_roi_saliency_batched(graphs[:2], (0, 1)))


def _attempt(case, fn):
    try:
        res = fn()
    except ValueError as e:
        case.outputs.update(str(e).encode())
        return
    for t in (res if isinstance(res, tuple) else (res,)):
        case.add(t)


def run_attribution_cases(shim, name, model, graphs, steps, points_per_pass, occlusions_per_pass, dump):
    """Integrated gradients with the completeness gap at each points_per_pass, then ROI occlusion at each
    occlusions_per_pass, both for classes (0, 1): one case each, outputs hashed."""
    with Case(shim) as case:
        for p in points_per_pass:
            _attempt(case, lambda: model.compute_integrated_gradients_batched(graphs, (0, 1), steps=steps,
                                                                              points_per_pass=p, return_delta=True))
    report(name + ".ig", case, dump)
    with Case(shim) as case:
        for o in occlusions_per_pass:
            _attempt(case, lambda: model.compute_roi_occlusion_batched(graphs, (0, 1), occlusions_per_pass=o))
    report(name + ".occlusion", case, dump)


def cpu_cases(dump):
    import emul_ops
    from helpers import Golden, SEED0, build_model, golden_names
    shim = TracingOps(emul_ops)
    for m in USERS:
        m._ops = shim
    engine.require_cuda = lambda dev: None
    torch.set_num_threads(1)
    names = [n for n in golden_names() if Golden(n).cfg["N"] < 400]
    for switch in (None, "FORCE_CSR_AGGREGATE", "FORCE_UNFUSED_BACKWARD"):
        if switch:
            setattr(engine, switch, True)
        for name in names:
            g = Golden(name)
            with Case(shim) as case:
                # under max pooling the dummy row is a batch-wide minimum: ROI averages one graph at a time, as the
                # reference's maps are per graph
                run_model_cases(case, build_model(g), g.graphs(), g.cfg["beta"], 4242 + SEED0[name],
                                roi_per_graph=g.cfg["neighbor_pooling_type"] == "max")
            report(name + ("." + switch if switch else ""), case, dump)
        if switch:
            setattr(engine, switch, False)
    g = Golden("tiny_eps_sum")
    graphs = g.graphs()
    for gr in graphs:
        gr.node_features = gr.node_features.clone()
        gr.node_features[0, 0] = 1.0000001          # not exactly one-hot: the dense layer-0 path
    with Case(shim) as case:
        run_model_cases(case, build_model(g), graphs, g.cfg["beta"], 7)
    report("tiny_eps_sum.dense_input", case, dump)
    # 6 points: 4 per pass splits each graph's points 4 + 2, 13 per pass packs two graphs; 7 copies per pass split every
    # graph's tags over several passes, 40 pack two small graphs or split one of 48 tags in two
    for name in names:
        g = Golden(name)
        run_attribution_cases(shim, name, build_model(g, g.state_after_train()), g.graphs(), 6, (4, 13), (7, 40), dump)


def gpu_cases(dump):
    from graph_neural_mapping_b200 import ops
    shim = TracingOps(ops)
    for m in USERS:
        m._ops = shim
    dev = torch.device("cuda")

    def model_of(layers, d, f, learn_eps=False, graph_pool="sum", nb_pool="sum", seed=0):
        torch.manual_seed(seed)
        m = GIN_InfoMaxReg(layers, 2, d, f, 2, 0.5, learn_eps, graph_pool, nb_pool, dev).to(dev)
        m.use_cuda_graphs = False
        return m

    def train_case(name, model, graphs, seed=5):
        with Case(shim) as case:
            c_logit, d_logit = _train_step(model, graphs, 0.05, seed)
            torch.cuda.synchronize()
            case.add(c_logit)
            case.add_grads(model)
        report(name, case, dump)

    def saliency_case(name, model, graphs, roi_graphs=None):
        with Case(shim) as case:
            case.add(model.compute_saliency_batched(graphs, 1))
            case.add(model.compute_roi_saliency_batched(roi_graphs or graphs, (0, 1)))
            torch.cuda.synchronize()
        report(name, case, dump)

    for fused in (True, False):
        model = model_of(5, 400, 64, seed=1)
        tr = driver.Trainer(model, fused=fused)
        graphs = synth.make_graphs_bulk(256, 400, 30, 128, seed0=10, device=dev)
        for step in range(4):                              # two eager warm-up steps, capture, replay
            np.random.seed(step)
            with Case(shim) as case:
                case.add(tr.step(graphs).reshape(1))
                torch.cuda.synchronize()
            report("trainer.fused=%s.step%d" % (fused, step), case, dump)

    model = model_of(5, 400, 64, seed=7)
    model.use_cuda_graphs = True
    for step in range(3):                                  # eager first sighting, capture, replay
        train_case("model.graphed.step%d" % step, model, graphs, seed=step)

    big = synth.make_graphs_bulk(1024, 400, 30, 128, seed0=20, device=dev)
    model = model_of(5, 400, 64, seed=2)
    train_case("model.1024x400", model, big)
    saliency_case("saliency.onehot.1024x400", model, big)
    # 8 points: 5 per pass splits each graph's points 5 + 3, 20 per pass packs two graphs; at 400 tags 300 copies per
    # pass split a graph's tags in two, 1024 pack two graphs
    attribution = dict(steps=8, points_per_pass=(5, 20), occlusions_per_pass=(300, 1024), dump=dump)
    run_attribution_cases(shim, "attribution.1024x400", model, big[:16], **attribution)
    dense = [synth.SynthGraph(400, g.label, g.edge_mat, g.node_features.clone()) for g in big[:64]]
    for gr in dense:
        gr.node_features[0, 0] = 0.5                          # not exactly one-hot: the dense layer-0 path
    saliency_case("roi.dense_input", model, dense)
    del big, dense

    small = synth.make_graphs(16, n_rois=64, n_time=128, seed0=30)
    train_case("learn_eps", model_of(3, 64, 64, learn_eps=True, seed=3), small)

    iso = synth.make_graphs(8, n_rois=64, n_time=128, seed0=40)
    em = iso[0].edge_mat
    iso[0].edge_mat = em[:, (em != 5).all(0)].contiguous()   # node 5 loses every neighbour (no self loop: learn_eps)
    model = model_of(3, 64, 64, learn_eps=True, nb_pool="average", graph_pool="average", seed=4)
    train_case("average.isolated", model, iso)
    saliency_case("average.isolated.saliency", model, iso)
    run_attribution_cases(shim, "average.isolated.attribution", model, iso, **attribution)

    mx = synth.make_graphs(8, n_rois=64, n_time=128, seed0=50, with_neighbors=True)
    model = model_of(3, 64, 64, nb_pool="max", seed=5)
    train_case("max", model, mx)
    saliency_case("max.saliency", model, mx[:1], roi_graphs=mx[:1])
    run_attribution_cases(shim, "max.attribution", model, mx, **attribution)

    wide = synth.make_graphs(16, n_rois=64, n_time=128, seed0=60)
    model = model_of(3, 64, 128, seed=6)
    train_case("hidden128", model, wide)
    saliency_case("hidden128.saliency", model, wide)
    run_attribution_cases(shim, "hidden128.attribution", model, wide, **attribution)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=["cpu", "gpu"])
    ap.add_argument("--dump", default=None, help="directory for the full traces")
    a = ap.parse_args()
    if a.dump:
        os.makedirs(a.dump, exist_ok=True)
    (cpu_cases if a.mode == "cpu" else gpu_cases)(a.dump)


if __name__ == "__main__":
    main()
