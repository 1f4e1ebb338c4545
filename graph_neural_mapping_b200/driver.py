"""Batched training driver beside the reference's frozen `main.py` (SURVEY 8(f) row N2).

`main.py:25-43` per step: `model(batch_graph)`, labels built on the host, CrossEntropy + beta * BCEWithLogits,
`zero_grad`, `backward`, `Adam.step`, `loss.cpu()`. Driven through the drop-in classes that loop already runs the
encoder from two CUDA graphs; what is left between them - prediction heads, loss, autograd bookkeeping, gradient
averaging, the optimizer - is ~100 small launches issued from Python every step.

`Trainer.step(batch_graph)` runs the WHOLE step - batch assembly kernel, encoder + DGI forward, heads, loss, backward,
data-parallel gradient averaging, Adam - as ONE captured CUDA graph per batch shape:

  per step (host):  batch assembly arithmetic (numpy gathers over the graph store's slot table), one permutation draw,
                    4 small asynchronous H2D copies through a pinned ring, one graph replay. No synchronisation: the
                    loss stays on the device (`.item()` it when you want to look at it).

Same arithmetic as the reference loop: the captured work is `engine.run_forward` / `run_backward` (the kernels of the
drop-in model), torch's own loss functions and `torch.optim.Adam(capturable=True)`; dropout uses torch's CUDA-graph
aware Philox generator. The first two steps of a new shape run eagerly (they warm up cuBLAS, the allocator and - data
parallel - NCCL), the third captures.
"""
import numpy as np
import torch

from . import dist as _dist
from . import engine as _engine
from . import graphed as _graphed
from . import ops as _ops


class _WholeStepPlan(object):
    def __init__(self, trainer, h, key, n_global):
        model = trainer.model
        dev = model.eps.device
        self.trainer, self.dev = trainer, dev
        self.inputs = _graphed.StepInputs(model, h, key, n_global, labels=True)
        self.d_labels = torch.cat([torch.ones(h.m, 1), torch.zeros(h.m, 1)], 0).to(dev)      # main.py:32-33
        self.graph = None
        self.loss = None
        self.launches = 0
        if trainer.fused:
            heads = list(model.linears_prediction)
            n_cls, n_feat = heads[0].weight.shape
            self.loss_terms = torch.zeros(2, dtype=torch.float64, device=dev)
            self.loss_out = torch.zeros(1, dtype=torch.float32, device=dev)
            self.heads_ws = torch.empty(_ops.heads_ce_workspace(h.b, len(heads), n_feat, n_cls), dtype=torch.float32, device=dev)
            self.heads_counter = torch.zeros(1, dtype=torch.int32, device=dev)
            self.c_logit = None

    def body(self):
        return self.body_fused() if self.trainer.fused else self.body_autograd()

    def body_fused(self):
        """One training step without torch autograd / torch.optim / torch loss kernels: encoder + DGI forward
        (engine.run_forward), prediction heads + dropout + CrossEntropy forward and backward (gnm_heads_ce),
        BCEWithLogits forward and backward (in the scoring pass of run_forward, or gnm_bce_logits where that kernel does
        not take the shape), the hand-derived backward (engine.run_backward),
        gradient averaging and Adam (gnm_adam_step). Same arithmetic as main.py:31-41."""
        tr = self.trainer
        model = tr.model
        dev = self.dev
        bs = self.inputs.structure()
        enc_params = _engine.flat_params(model)
        params = [p.detach() for p in enc_params]
        b, m = bs.n_graphs, bs.n_rows
        self.loss_terms.zero_()                     # [CE mean, beta * BCE mean], float64
        w_bce = tr.beta / (2.0 * m)                 # main.py:32-37: BCEWithLogits mean over 2m scores, times beta
        g_f, d_logit, sv = _engine.run_forward(model, bs, self.inputs.neg_idx, True, True, None, params, tr.comm,
                                               bce=(w_bce, w_bce, self.loss_terms[1:2]))
        heads = list(model.linears_prediction)
        n_layers, n_cls, n_feat = len(heads), heads[0].weight.shape[0], heads[0].weight.shape[1]
        hw = [h.weight.detach() for h in heads]
        hb = [h.bias.detach() for h in heads]
        d_hw = [torch.empty_like(w) for w in hw]
        d_hb = [torch.empty_like(x) for x in hb]
        mask = None
        if model.final_dropout > 0.0:
            # F.dropout's keep mask (graphcnn.py:230), one draw for all layers from torch's (CUDA-graph aware) generator
            keep = 1.0 - float(model.final_dropout)
            mask = torch.empty(n_layers, b, n_cls, dtype=torch.float32, device=dev).bernoulli_(keep).mul_(1.0 / keep)
        c_logit = torch.empty(b, n_cls, dtype=torch.float32, device=dev)
        d_gf = torch.empty_like(g_f)
        _ops.heads_ce(g_f, hw, hb, mask, self.inputs.labels, 1.0 / b, c_logit, self.loss_terms[0:1], d_gf, d_hw, d_hb,
                      self.heads_ws, self.heads_counter)
        dd = None
        if sv.scored is None:
            # the scoring kernel did not take this shape: BCE forward and backward on the scores here
            dd = torch.empty(2 * m, 1, dtype=torch.float32, device=dev)
            _ops.bce_logits(d_logit.view(-1), m, w_bce, w_bce, self.loss_terms[1:2], dd.view(-1))
        _, enc_grads = _engine.run_backward(model, sv, params, d_gf, dd, False, tr.comm)
        tensors, grads = [], []
        for p, g in zip(enc_params, enc_grads):
            if g is not None and p.requires_grad:
                tensors.append(p)
                grads.append(g.reshape(p.shape))
        for h, gw, gb in zip(heads, d_hw, d_hb):
            tensors += [h.weight, h.bias]
            grads += [gw, gb]
        grad_scale = 1.0
        world = tr.comm.world
        if world > 1:
            # one flat all-reduce; each rank's loss is the mean over its own shard, so the average over ranks is the
            # gradient of the global-batch mean loss (main.py:34-41 at the global batch)
            flat = torch.cat([g.reshape(-1) for g in grads])
            tr.comm.all_reduce_mean_flat(flat)
            views, off = [], 0
            for g in grads:
                views.append(flat[off:off + g.numel()].view(g.shape))
                off += g.numel()
            grads = views
        state = tr.adam_state(tensors)
        group = tr.optimizer.param_groups[0]
        _ops.adam_step([p.detach() for p in tensors], [g.contiguous() for g in grads], state["offsets"], state["exp_avg"],
                       state["exp_avg_sq"], state["step"], group["lr"], group["betas"][0], group["betas"][1], group["eps"],
                       group["weight_decay"], grad_scale, loss_terms=self.loss_terms, loss_out=self.loss_out)
        for p, g in zip(tensors, grads):
            p.grad = g                                   # for inspection (aliases step-local / CUDA-graph memory)
        self.c_logit = c_logit
        return self.loss_out[0]

    def body_autograd(self):
        """One training step on the static buffers (runs eagerly while warming up, then under capture)."""
        tr = self.trainer
        model = tr.model
        runner = _engine.Runner(model, self.inputs.structure(), self.inputs.neg_idx, True, True, tr.comm)
        tr.optimizer.zero_grad(set_to_none=True)
        g_f, d_logit = _engine.GINFunction.apply(runner, None, *_engine.flat_params(model))
        c_logit = model._heads(g_f)
        loss = tr.c_criterion(c_logit, self.inputs.labels) +tr.beta * tr.d_criterion(d_logit, self.d_labels)     # main.py:34-37
        loss.backward()
        _dist.average_gradients(model, tr.comm)
        tr.optimizer.step()
        return loss.detach()

    def run(self):
        if self.graph is None:
            self.graph, self.loss, self.launches = _graphed.capture(self.body)
        _graphed.replay(self.graph, self.launches)
        return self.loss


class Trainer(object):
    """`main.py:25-43` as one CUDA graph per batch shape. `model` is a `GIN_InfoMaxReg` in train mode on a CUDA device
    with one-hot node features; `comm` the data-parallel communicator (`dist.init_from_env()`), each rank passing its
    own shard of the global batch. Adam only (the reference's optimizer, `main.py:137`)."""

    def __init__(self, model, lr=0.005, beta=0.05, comm=None, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0,
                 check_every=100, fused=True):
        """Defaults follow main.py:113,118 (--lr 0.005, --beta 0.05). The learning rate lives in a DEVICE tensor, so
        a scheduler (`torch.optim.lr_scheduler.StepLR(trainer.optimizer, ...)`, main.py:138,147) or `set_lr()` changes
        what the captured step reads - a Python float would be baked into the CUDA graph at capture.
        `check_every`: every that many steps (and in `finish()`) the kernels' bounded-wait flags are polled (one device
        synchronisation); a tcgen05 pipeline or peer exchange that timed out raises instead of training on garbage."""
        dev = model.eps.device
        _engine.require_cuda(dev)
        self.model = model
        self.beta = float(beta)
        self.comm = comm if comm is not None else _dist.SINGLE
        model.set_comm(self.comm)
        self.optimizer = torch.optim.Adam(model.parameters(), lr=torch.tensor(float(lr), dtype=torch.float32, device=dev),
                                          betas=betas, eps=eps, weight_decay=weight_decay, capturable=True)
        self.check_every = int(check_every)
        self.steps_done = 0
        # fused=True: the step's [B, L*F]-sized remainder (heads, dropout, CE, BCE, Adam) runs on libgnm's own kernels
        # (gnm_train.cu) and the backward is called directly - no torch autograd / loss / optimizer kernels in the
        # step. fused=False: torch's loss functions, autograd and torch.optim.Adam(capturable=True) around the same
        # encoder kernels (the round-1 driver; kept as the A/B reference of the fused path).
        self.fused = bool(fused)
        self._adam = None
        self.c_criterion = torch.nn.CrossEntropyLoss()          # main.py:16
        self.d_criterion = torch.nn.BCEWithLogitsLoss()         # main.py:17
        self._plans = {}
        self._seen = {}
        self.h2d_bytes = 0

    def adam_state(self, tensors):
        """Flat Adam moments shared with `self.optimizer.state` (so `optimizer.state_dict()` checkpoints them and a
        later `optimizer.step()` would continue from them): created on first use for exactly the parameters that
        receive gradients, like torch.optim.Adam's lazy state initialisation."""
        ids = tuple(id(p) for p in tensors)
        if self._adam is not None and self._adam["ids"] == ids:
            return self._adam
        if self._adam is not None:
            raise RuntimeError("the set of parameters receiving gradients changed between steps")
        dev = tensors[0].device
        offsets, total = [], 0
        for p in tensors:
            offsets.append(total)
            total += (p.numel() + 3) // 4 * 4
        st = {"ids": ids, "offsets": offsets, "exp_avg": torch.zeros(total, dtype=torch.float32, device=dev),
              "exp_avg_sq": torch.zeros(total, dtype=torch.float32, device=dev),
              "step": torch.zeros(2, dtype=torch.float32, device=dev)}
        for p, off in zip(tensors, offsets):
            n = p.numel()
            self.optimizer.state[p] = {"step": st["step"][0], "exp_avg": st["exp_avg"][off:off + n].view_as(p),
                                       "exp_avg_sq": st["exp_avg_sq"][off:off + n].view_as(p)}
        self._adam = st
        return st

    def set_lr(self, lr):
        """Change the learning rate of every parameter group in place (visible to the captured CUDA graph)."""
        for group in self.optimizer.param_groups:
            if torch.is_tensor(group["lr"]):
                group["lr"].fill_(float(lr))
            else:
                group["lr"] = float(lr)

    def get_lr(self):
        return float(self.optimizer.param_groups[0]["lr"])

    def check(self):
        """Poll the kernels' bounded-wait flags (synchronises the device). Raises if a tcgen05 kernel or a peer-memory
        exchange gave up waiting since the last check: every step since then is invalid."""
        if _ops.aggregate_tc_status():
            raise RuntimeError("a tcgen05 kernel (aggregation / linear) hit its bounded barrier wait: the steps since "
                               "the last check are invalid")
        p2p = self.comm.p2p
        if p2p is not None and p2p.status():
            raise RuntimeError("a peer-memory exchange gave up waiting for a peer: BatchNorm statistics (and everything "
                               "after them) were poisoned with NaN on this rank")

    def finish(self):
        """Call at the end of training / an epoch: drains the stream and checks the kernels' status flags."""
        torch.cuda.synchronize(self.model.eps.device)
        self.check()

    def release(self):
        """Drop the captured graphs (do this before tearing a process group down: they hold NCCL work)."""
        self._plans.clear()
        self._seen.clear()

    def step(self, batch_graph, labels=None):
        """One optimisation step on `batch_graph` (this rank's shard). Returns the loss as a 0-d device tensor that is
        overwritten by the next step of the same shape; nothing synchronises."""
        model = self.model
        if not model.training:
            raise RuntimeError("Trainer.step needs model.train()")
        n_global = len(batch_graph) * self.comm.world
        perm = np.random.permutation(n_global)                  # graphcnn.py:199: one numpy draw per step
        h = model._host_batch(batch_graph)
        if h.uniform_n is None:
            raise RuntimeError("GIN_InfoMaxReg needs graphs with the same number of nodes (graphcnn.py:198-201)")
        if not h.onehot or (model.neighbor_pooling_type == "max" and not h.max0_as_sum):
            raise RuntimeError("Trainer runs the one-hot input path (util.py:114-116); use the model API for dense features")
        if labels is None:
            labels = [g.label for g in batch_graph]             # main.py:31
        key = _graphed.plan_key(h, n_global, self.comm.world)
        plan = self._plans.get(key)
        if plan is not None and not plan.inputs.fits(h, key):
            del self._plans[key]
            plan = None
        if plan is None:
            while len(self._plans) >= 2:
                self._plans.pop(next(iter(self._plans)))
            plan = _WholeStepPlan(self, h, key, n_global)
            self._plans[key] = plan
            self._seen[key] = 0
        self.h2d_bytes += plan.inputs.load(h, perm, labels)
        self._seen[key] += 1
        self.steps_done += 1
        if self.check_every > 0 and self.steps_done % self.check_every == 0:
            self.check()
        if self._seen[key] <= 2:
            return plan.body()                                   # warm-up: cuBLAS handles, allocator, NCCL
        return plan.run()


# ------------------------------------------------------------------------------------------------------------------
# Batched evaluation: main.py:49-82 runs its three evaluation loops one graph per forward (`model([g])`). In eval mode
# BatchNorm uses the running statistics and Adj_block is block-diagonal, so class logits, the latent space and the
# saliency maps of a graph do not depend on its batch companions: the loops below produce the same arrays, in the same
# layout, from large batches (SURVEY 8(f) N1 / N3).
# ------------------------------------------------------------------------------------------------------------------

def _batches(graphs, batch):
    for i in range(0, len(graphs), batch):
        yield graphs[i:i + batch]


def class_logits(model, graphs, batch=256):
    """`pass_data_iteratively(model, graphs)[0]` (main.py:49-57): [G, 2] class logits, eval mode, on the device."""
    model.eval()
    out = []
    with torch.no_grad():
        for chunk in _batches(graphs, batch):
            if len({len(g.g) for g in chunk}) > 1:
                out.extend(model([g])[0] for g in chunk)         # ragged node counts: the DGI path needs equal sizes
            else:
                out.append(model(chunk)[0])
    return torch.cat(out, 0)


def latent_space(model, graphs, batch=256):
    """`get_latent_space` (main.py:71-82): (float32 [G, L*F] readout features, int [G, 1] labels)."""
    model.eval()
    feats = []
    with torch.no_grad():
        for chunk in _batches(graphs, batch):
            if len({len(g.g) for g in chunk}) > 1:
                feats.extend(model([g], latent=True) for g in chunk)
            else:
                feats.append(model(chunk, latent=True))
    labels = np.stack([np.array([g.label]) for g in graphs], axis=0)
    return np.concatenate(feats, axis=0), labels


def stream_saliency(model, graphs, cls, sink, batch=64):
    """Batched `compute_saliency` (exact, SURVEY A10) streamed to `sink(first_graph, array)`: the maps of one batch
    ([b, N, D] float32 numpy view of a PINNED host buffer, valid until the call after next) are handed over while the
    device already computes the next batch - two pinned buffers, asynchronous D2H, one event each. Nothing accumulates:
    100k graphs x 640 KB never sit in host RAM unless the sink keeps them."""
    dev = model.eps.device
    bufs, events = [None, None], [None, None]
    pending = None                          # (slot, first graph index, shape) of the batch whose copy is in flight
    i0 = 0

    def flush(p):
        slot, first, shape = p
        if events[slot] is not None:
            events[slot].synchronize()
        n_el = int(np.prod(shape))
        sink(first, bufs[slot][:n_el].numpy().reshape(shape))

    for k, chunk in enumerate(_batches(graphs, batch)):
        s = model.compute_saliency_batched(chunk, cls).detach()
        n = len(chunk[0].g)
        shape = (len(chunk), n, int(s.shape[1]))
        slot = k & 1
        if bufs[slot] is None or bufs[slot].numel() < s.numel():
            bufs[slot] = torch.empty(s.numel(), dtype=torch.float32, pin_memory=(dev.type == "cuda"))
            events[slot] = torch.cuda.Event() if dev.type == "cuda" else None
        bufs[slot][:s.numel()].copy_(s.reshape(-1), non_blocking=True)
        if events[slot] is not None:
            events[slot].record()
        if pending is not None:
            flush(pending)                  # the previous batch: its copy overlapped this batch's kernels
        pending = (slot, i0, shape)
        i0 += len(chunk)
    if pending is not None:
        flush(pending)
    return i0


def saliency_maps(model, graphs, cls, batch=64):
    """`get_saliency_map` (main.py:60-68): float32 [G, N, D] - one `compute_saliency` map per graph, computed in
    batches (exact: `compute_saliency_batched`). All graphs must have the same number of nodes (np.stack)."""
    out = {}

    def sink(first, arr):
        if "a" not in out:
            out["a"] = np.empty((len(graphs),) + arr.shape[1:], dtype=np.float32)
        out["a"][first:first + arr.shape[0]] = arr
    stream_saliency(model, graphs, cls, sink, batch)
    return out.get("a", np.zeros((0, 0, 0), dtype=np.float32))


def _attribution_chunks(model, graphs, classes, batch, compute, with_delta=False):
    """compute(chunk) on `graphs` in chunks of `batch` graphs, one D2H copy per chunk: float32 [G, len(classes), D] from
    its [n, len(classes), D] device results, and with_delta also [G, len(classes)] from a second result."""
    c, d = len(classes), int(_engine.layer_units(model, 0)[0][0].weight.shape[1])          # d: input_dim
    width = c * d + (c if with_delta else 0)
    host = np.empty((len(graphs), width), dtype=np.float32)
    for i in range(0, len(graphs), batch):
        chunk = graphs[i:i + batch]
        res = compute(chunk)
        flat = torch.cat([res[0].reshape(len(chunk), c * d), res[1]], 1) if with_delta else res.reshape(len(chunk), width)
        host[i:i + len(chunk)] = flat.cpu().numpy()                    # one copy for both results
    out = np.ascontiguousarray(host[:, :c * d]).reshape(len(graphs), c, d)
    return (out, np.ascontiguousarray(host[:, c * d:])) if with_delta else out


def roi_saliency(model, graphs, classes=(0, 1), batch=1024):
    """ROI saliency: float32 [G, len(classes), D], entry [i, k] = the node average of `compute_saliency([graphs[i]],
    classes[k])` - what evaluate/plot_saliency_nii.py reduces each map to - computed by
    `compute_roi_saliency_batched` in batches of `batch` graphs (one forward per batch for all classes, one D2H copy
    per batch; 1.6 KB per graph and class instead of a 640 KB map at N = D = 400). Graphs may differ in size."""
    return _attribution_chunks(model, graphs, classes, batch,
                               lambda chunk: model.compute_roi_saliency_batched(chunk, classes))


def integrated_gradients(model, graphs, classes=(0, 1), steps=50, batch=1024, return_delta=False):
    """Integrated gradients (zero baseline, midpoint rule with `steps` points): float32 [G, len(classes), D], entry
    [i, k] = the node average of graph i's attribution map for classes[k] (`compute_integrated_gradients_batched`, the
    same node average as `roi_saliency`), and with return_delta the [G, len(classes)] completeness gap. Computed in
    calls of `batch` graphs, one D2H copy per call. Graphs may differ in size; node features must be one-hot and the
    neighbour pooling sum or average."""
    return _attribution_chunks(model, graphs, classes, batch, lambda chunk: model.compute_integrated_gradients_batched(
        chunk, classes, steps=steps, return_delta=return_delta), return_delta)


def roi_occlusion(model, graphs, classes=(0, 1), batch=1024):
    """ROI occlusion (zero baseline): float32 [G, len(classes), D], entry [i, k, d] = (F_c(X_i) - F_c(X_i with column d
    set to 0)) / n_i for c = classes[k] (`compute_roi_occlusion_batched`, the node-average convention of `roi_saliency`
    and `integrated_gradients`). Computed in calls of `batch` graphs, one D2H copy per call. Graphs may differ in size;
    node features must be one-hot, and under max neighbour pooling tags injective and edge lists duplicate-free."""
    return _attribution_chunks(model, graphs, classes, batch,
                               lambda chunk: model.compute_roi_occlusion_batched(chunk, classes))


def saliency_maps_to_npy(model, graphs, cls, path, batch=64):
    """`np.save(path, get_saliency_map(model, graphs, cls))` (main.py:168-172) without holding the array: the `.npy`
    file is created as a memory map of its final shape [G, N, D] and filled batch by batch from the pinned double
    buffer. Same bytes on disk as the reference's np.save (format 1.0/2.0 header + C-order float32)."""
    n, d = len(graphs[0].g), int(graphs[0].node_features.shape[1])
    mm = np.lib.format.open_memmap(path, mode="w+", dtype=np.float32, shape=(len(graphs), n, d))

    def sink(first, arr):
        mm[first:first + arr.shape[0]] = arr
    stream_saliency(model, graphs, cls, sink, batch)
    mm.flush()
    del mm
    return path


def save_results(model, graphs, out_dir, batch=64):
    """The arrays main.py:170-172 leaves for the evaluate/ scripts, same file names and layouts: latent_space.npy,
    labels.npy, saliency_female.npy (class 0), saliency_male.npy (class 1). The saliency files are streamed
    (saliency_maps_to_npy): host memory stays at two batches however many graphs there are."""
    import os
    os.makedirs(out_dir, exist_ok=True)
    lat, labels = latent_space(model, graphs, batch=max(batch, 1))
    np.save(os.path.join(out_dir, "latent_space.npy"), lat)
    np.save(os.path.join(out_dir, "labels.npy"), labels)
    saliency_maps_to_npy(model, graphs, 0, os.path.join(out_dir, "saliency_female.npy"), batch)
    saliency_maps_to_npy(model, graphs, 1, os.path.join(out_dir, "saliency_male.npy"), batch)
    return out_dir
