"""CUDA-graph execution of the training step's encoder forward / backward.

A training step launches ~130 libgnm kernels plus a few dozen small torch ops; issued one by
one from Python they leave the B200 idle between launches (host-bound: 14-30 ms per step for
11 ms of kernels in the first measurements). The shapes of a training step are static
(B graphs of N nodes), so `engine.run_forward` / `engine.run_backward` - the same Python
orchestration, unchanged - are captured ONCE per shape into two CUDA graphs and replayed:

  per step (host):  3 small H2D copies (slot addresses, node offsets, DGI permutation)
                    -> forward graph replay -> [driver: heads, loss, autograd]
                    -> 2 D2D copies of the incoming gradients -> backward graph replay

Inputs and outputs live in static buffers owned by the plan; outputs and gradients are
cloned before they are handed to autograd so the caller never aliases graph memory.
BatchNorm running statistics, NCCL all-reduces (data parallel) and the batch assembly kernel
are part of the captured work.

driver.Trainer captures its whole step as one graph on the same pieces: the plan key, the
check that a plan still fits a batch and the static inputs with their pinned ring
(StepInputs), and capture / replay with the launch accounting.
"""
import torch

from . import engine as _engine
from . import ops as _ops


import contextlib
import gc


@contextlib.contextmanager
def quiet_capture():
    """Around a CUDA-graph capture: Python's cyclic garbage collector must not run inside it. Collecting an old plan
    (a CUDAGraph with its private memory pool, pinned staging buffers) calls cudaGraphExecDestroy / cudaFree-class APIs,
    which are not permitted while a stream is capturing and invalidate the capture ("operation not permitted when
    stream is capturing" at capture_end, seen once in a long test process). Collect first, then hold the collector."""
    gc.collect()
    was_enabled = gc.isenabled()
    gc.disable()
    try:
        yield
    finally:
        if was_enabled:
            gc.enable()


def plan_key(h, n_global, world):
    """What a captured step bakes in from host batch `h` through its kernel choices and buffer shapes, with `n_global`
    DGI negatives over `world` data-parallel ranks: batches with equal keys can replay one plan (StepInputs.fits)."""
    return (h.b, h.m, h.uniform_n, h.onehot, h.feat_dim, h.n_max, h.dense, h.has_isolated, h.same_tags, h.max0_as_sum,
            n_global, world)


def _pointers(model):
    return list(map(torch.Tensor.data_ptr, _engine.flat_params(model) + _engine.flat_buffers(model)))


class StepInputs(object):
    """The static inputs of a captured training step - the batch's slot addresses / offsets (`packed`, `node_off`), the
    DGI permutation (`neg_idx`) and, with `labels`, the class labels - refilled by load() before every step. Also keeps
    what else the graph bakes in: the plan key, the capacity of the batch CSR and the addresses of the model's
    parameters and BatchNorm buffers when the plan was made."""

    def __init__(self, model, h, key, n_neg, labels=False):
        dev = model.eps.device
        self.model, self.key, self.h = model, key, h
        self.nnz_cap = int(h.nnz * 1.02) + 4096
        self.ptrs = _pointers(model)
        self.packed = torch.zeros(5 * h.b + 1, dtype=torch.int64, device=dev)
        self.node_off = torch.zeros(h.b + 1, dtype=torch.int32, device=dev)
        self.neg_idx = torch.zeros(n_neg, dtype=torch.int32, device=dev)
        self.labels = torch.zeros(h.b, dtype=torch.int64, device=dev) if labels else None
        self._dst = [t for t in (self.packed, self.node_off, self.neg_idx, self.labels) if t is not None]
        self._stage = [None, None, None]
        self._stage_i = 0

    def fits(self, h, key):
        """Whether a step on host batch `h` with plan key `key` may replay the plan: same key, nnz within the capacity,
        and the model's parameters and BatchNorm buffers still where they were. Replacing a buffer tensor
        (`bn.running_mean = bn.running_mean.clone()`, load_state_dict(assign=True) + release_graphs()) moves it: a
        replay would update the tensor the model no longer holds."""
        return key == self.key and h.nnz <= self.nnz_cap and _pointers(self.model) == self.ptrs

    def load(self, h, perm, labels=None):
        """Per-step host -> device traffic: slot addresses / offsets, the DGI permutation and the labels, staged through
        a small ring of pinned buffers and copied asynchronously, so the host never waits for the previous step's
        kernels and can prepare (and enqueue) the next step while the GPU is still busy with this one. Returns the
        bytes shipped."""
        self.h = h
        i = self._stage_i
        self._stage_i = (i + 1) % len(self._stage)
        if self._stage[i] is None:
            self._stage[i] = ([torch.empty(t.shape[0], dtype=t.dtype, pin_memory=True) for t in self._dst],
                              torch.cuda.Event())
        else:
            self._stage[i][1].synchronize()           # the copies that last read this slot (three steps ago) are done
        pinned, ev = self._stage[i]
        for s, x in zip(pinned, (h.packed, h.node_off, perm, labels)):
            s.numpy()[:] = x
        for t, s in zip(self._dst, pinned):
            t.copy_(s, non_blocking=True)
        ev.record()
        return sum(s.nbytes for s in pinned)

    def structure(self):
        """The BatchStructure of the loaded batch, gathered from the static buffers (also under capture)."""
        model = self.model
        return model._graph_store().assemble(self.h, model.graph_pooling_type, self.packed, self.node_off, self.nnz_cap)


def capture(body, pool=None):
    """body() captured into a CUDA graph in memory pool `pool` (None: a private one). Returns (graph, body's result,
    libgnm kernels recorded). Capture records the kernels without running them, so they come off ops.REPLAYED here and
    replay() adds them back whenever they run."""
    g = torch.cuda.CUDAGraph()
    n0 = _ops.kernels_recorded()
    with quiet_capture(), torch.cuda.graph(g, pool=pool):
        out = body()
    launches = _ops.kernels_recorded() - n0           # libgnm kernels inside the graph (C-side counters)
    _ops.REPLAYED[0] -= launches
    return g, out, launches


def replay(graph, launches):
    graph.replay()
    _ops.REPLAYED[0] += launches


class StepPlan(object):
    """Captured encoder forward and backward graphs, in one memory pool, for one training-step shape."""

    def __init__(self, model, host_batch, key, n_neg, comm):
        self.model, self.comm = model, comm
        self.inputs = StepInputs(model, host_batch, key, n_neg)
        self.pool = torch.cuda.graph_pool_handle()
        self.fwd_graph = None
        self.bwd_graph = None
        self.generation = 0

    def forward(self):
        if self.fwd_graph is None:
            model, inputs = self.model, self.inputs
            self.params = [p.detach() for p in _engine.flat_params(model)]
            self.fwd_graph, (self.g_f, self.d_logit, self.sv), self.fwd_launches = capture(
                lambda: _engine.run_forward(model, inputs.structure(), inputs.neg_idx, True, True, None, self.params,
                                            self.comm), self.pool)
        replay(self.fwd_graph, self.fwd_launches)
        self.generation += 1
        return self.g_f.clone(), self.d_logit.clone()

    def _backward_body(self):
        _, grads = _engine.run_backward(self.model, self.sv, self.params, self.dg_in, self.dd_in, False, self.comm)
        self.grad_shapes = [None if x is None else tuple(x.shape) for x in grads]
        self.grad_sizes = [int(x.numel()) for x in grads if x is not None]
        return torch.cat([x.reshape(-1) for x in grads if x is not None])

    def backward(self, dg_f, dd_logit):
        if self.bwd_graph is None:
            self.dg_in = torch.zeros_like(self.g_f)
            self.dd_in = torch.zeros_like(self.d_logit)
        self.dg_in.copy_(dg_f)
        self.dd_in.copy_(dd_logit)
        if self.bwd_graph is None:
            self.bwd_graph, self.flat, self.bwd_launches = capture(self._backward_body, self.pool)
        replay(self.bwd_graph, self.bwd_launches)
        pieces = iter(self.flat.clone().split(self.grad_sizes))        # one call: the per-tensor slicing was host time
        return [None if shp is None else next(pieces).view(shp) for shp in self.grad_shapes]


class GraphedGINFunction(torch.autograd.Function):
    """Same contract as engine.GINFunction, executed by replaying the plan's CUDA graphs."""

    @staticmethod
    def forward(ctx, plan, *params):
        g_f, d_logit = plan.forward()
        ctx.plan = plan
        ctx.generation = plan.generation
        ctx.params = params
        return g_f, d_logit

    @staticmethod
    def backward(ctx, dg_f, dd_logit):
        plan = ctx.plan
        if ctx.generation != plan.generation:
            raise RuntimeError("GIN_InfoMaxReg: backward() of an earlier forward was called after a newer forward of the "
                               "same shape; with CUDA graphs the activations live in static buffers. Call backward "
                               "before the next forward, or set model.use_cuda_graphs = False.")
        if dg_f is None:
            dg_f = torch.zeros_like(plan.g_f)
        if dd_logit is None:
            dd_logit = torch.zeros_like(plan.d_logit)
        grads = plan.backward(dg_f, dd_logit)
        out = [g if (g is not None and p.requires_grad) else None for p, g in zip(ctx.params, grads)]
        return (None,) + tuple(out)
