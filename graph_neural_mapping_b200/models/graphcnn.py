"""`GIN_InfoMaxReg` with the reference's constructor, `forward` / `compute_saliency`
signatures and state_dict layout (reference: models/graphcnn.py:12-299), executed by the
libgnm sm_100a kernels through `engine.GINFunction`.

What stays in Python here is exactly what the reference driver relies on:
  * one `np.random.permutation(len(batch_graph))` draw per forward (graphcnn.py:199),
  * the `(c_logit, d_logit)` / `latent=True` return contract (graphcnn.py:248-251),
  * `compute_saliency`'s side effects (`eval()`, `zero_grad()`, parameter `.grad`s).
The prediction heads (`linears_prediction` + dropout on [B, F] rows, graphcnn.py:230) are
[B, 2]-sized and stay in torch so the dropout mask comes from the same torch RNG stream as
the reference's.
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from .mlp import MLP
from .discriminator import Discriminator
import os

from .. import dist as _dist
from .. import engine as _engine
from .. import graphed as _graphed
from .. import ops as _ops


class _HeadsFunction(torch.autograd.Function):
    """c_logit = sum_l mask_l * (g_f[:, l] W_l^T + b_l) (graphcnn.py:228-231) on gnm_heads_fwd / gnm_heads_bwd."""

    @staticmethod
    def forward(ctx, g_f, mask, n_layers, *wb):
        from .. import ops as _ops
        ws = [w.detach().contiguous() for w in wb[:n_layers]]
        bs = [b.detach().contiguous() for b in wb[n_layers:]]
        g = g_f.detach()
        if g.stride(1) != 1:
            g = g.contiguous()
        c_logit = torch.empty(g.shape[0], ws[0].shape[0], dtype=torch.float32, device=g.device)
        _ops.heads_fwd(g, ws, bs, mask, c_logit)
        ctx.n_layers = n_layers
        ctx.mask = mask
        ctx.save_for_backward(g, *ws)
        return c_logit

    @staticmethod
    def backward(ctx, d_logit):
        from .. import ops as _ops
        g, ws = ctx.saved_tensors[0], list(ctx.saved_tensors[1:])
        n_cls, n_feat = ws[0].shape
        d_gf = torch.empty_like(g)
        dws = [torch.empty_like(w) for w in ws]
        dbs = [torch.empty(n_cls, dtype=torch.float32, device=g.device) for _ in ws]
        work = torch.empty(_ops.heads_ce_workspace(g.shape[0], ctx.n_layers, n_feat, n_cls), dtype=torch.float32, device=g.device)
        counter = torch.zeros(1, dtype=torch.int32, device=g.device)
        _ops.heads_bwd(g, ws, ctx.mask, d_logit.contiguous(), d_gf, dws, dbs, work, counter)
        return (d_gf, None, None) + tuple(dws) + tuple(dbs)


class GIN_InfoMaxReg(nn.Module):
    def __init__(self, num_layers, num_mlp_layers, input_dim, hidden_dim, output_dim, final_dropout, learn_eps,
                 graph_pooling_type, neighbor_pooling_type, device):
        super().__init__()
        # module creation order follows graphcnn.py:29-52 so torch.manual_seed(s) + constructor
        # yields the reference's initial weights
        self.disc = Discriminator(hidden_dim * num_layers)
        self.sigm = nn.Sigmoid()
        self.relu = nn.ReLU()

        self.final_dropout = final_dropout
        self.device = device
        self.num_layers = num_layers
        self.hidden_dim = hidden_dim
        self.graph_pooling_type = graph_pooling_type
        self.neighbor_pooling_type = neighbor_pooling_type
        self.learn_eps = learn_eps
        self.eps = nn.Parameter(torch.zeros(num_layers))

        self.mlps = nn.ModuleList()
        self.batch_norms = nn.ModuleList()
        self.linears_prediction = nn.ModuleList()
        for layer in range(num_layers):
            self.mlps.append(MLP(num_mlp_layers, input_dim if layer == 0 else hidden_dim, hidden_dim, hidden_dim))
            self.batch_norms.append(nn.BatchNorm1d(hidden_dim))
            self.linears_prediction.append(nn.Linear(hidden_dim, output_dim))

        self._store = None
        self._comm = _dist.SINGLE
        self.cache_graphs = True        # keep per-graph CSRs resident on the device between calls
        # training steps of a repeated shape are captured into CUDA graphs (graphed.py) after one eager warm-up
        self.use_cuda_graphs = os.environ.get("GNM_CUDA_GRAPHS", "1") != "0"
        self._plans = {}
        self._warm = set()

    # ---- data-parallel hook (new; the reference is single-process) -------------------------
    def set_comm(self, comm):
        """Engage data parallelism: `forward` then expects THIS rank's contiguous shard of the
        global batch and synchronises BatchNorm statistics and the DGI negatives over `comm`."""
        self._comm = comm if comm is not None else _dist.SINGLE

    def forget_graphs(self):
        """Drop the device-resident per-graph CSR cache (e.g. after editing a graph's `edge_mat` in place: the cache is
        keyed on the graph objects, SURVEY 8(b) ownership)."""
        if self._store is not None:
            self._store.clear()

    def release_graphs(self):
        """Drop the captured CUDA graphs (and their static buffers); they are re-captured on demand."""
        self._plans.clear()
        self._warm.clear()
        self.__dict__.pop("_gnm_flat_params", None)
        self.__dict__.pop("_gnm_flat_bns", None)

    def _apply(self, fn, *args, **kwargs):
        self.__dict__.pop("_gnm_flat_params", None)
        self.__dict__.pop("_gnm_flat_bns", None)
        return super()._apply(fn, *args, **kwargs)

    # ---- internals --------------------------------------------------------------------------
    def _graph_store(self):
        dev = self.eps.device
        _engine.require_cuda(dev)
        if self._store is None or self._store.device != dev or self._store.add_self_loops != (not self.learn_eps):
            self._store = _engine.GraphStore(dev, add_self_loops=not self.learn_eps)
        return self._store

    def _host_batch(self, batch_graph):
        if self.neighbor_pooling_type not in ("sum", "average", "max"):
            raise ValueError("unknown neighbor_pooling_type %r" % (self.neighbor_pooling_type,))
        store = self._graph_store()
        if not self.cache_graphs:
            store.clear()
        return store.assemble_host(batch_graph)

    def _structure(self, batch_graph, host_batch=None):
        h = host_batch if host_batch is not None else self._host_batch(batch_graph)
        return self._graph_store().assemble(h, self.graph_pooling_type)

    def _step_plan(self, h, n_global):
        """The CUDA-graph plan for this training-step shape, or None (first sighting runs eagerly: it warms up
        cuBLAS / NCCL and the allocator before capture)."""
        if not (self.use_cuda_graphs and self.training and torch.is_grad_enabled() and h.onehot
                and (self.neighbor_pooling_type != "max" or h.max0_as_sum) and self.eps.device.type == "cuda"):
            return None
        key = _graphed.plan_key(h, n_global, self._comm.world)          # training only: comm is self._comm
        plan = self._plans.get(key)
        if plan is not None and not plan.inputs.fits(h, key):
            del self._plans[key]
            plan = None
        if plan is None:
            if key not in self._warm:
                self._warm.add(key)
                return None
            while len(self._plans) >= 2:
                self._plans.pop(next(iter(self._plans)))
            plan = _graphed.StepPlan(self, h, key, n_global, self._comm)
            self._plans[key] = plan
        return plan

    def _dense_features(self, batch_graph, bs):
        if bs.onehot and (self.neighbor_pooling_type != "max" or bs.max0_as_sum):
            return None                 # layer 0 runs as a row gather of W1^T
        return torch.cat([g.node_features for g in batch_graph], 0).to(self.eps.device, torch.float32)

    def _padded_neighbours(self, batch_graph):
        """The padded neighbour lists of graphcnn.py:55-81 as global row ids ([M, W] int64, -1 pads; the node itself
        appended when learn_eps is False) and their first entries ([M], -1 where the list starts with a pad).
        torch.max breaks ties towards the first list entry, so input gradients under max pooling need the reference's
        neighbour ORDER: `graph.neighbors` (util.py:86-90) when the graph carries it, else rebuilt from `edge_mat`,
        whose first half lists the edges in the same order (util.py:99-103)."""
        lists = []
        for g in batch_graph:
            n = len(g.g)
            nb = getattr(g, "neighbors", None)
            if nb is None or len(nb) != n or not any(len(x) for x in nb):
                nb = [[] for _ in range(n)]
                em = g.edge_mat
                if torch.is_tensor(em) and em.numel() > 0:
                    e = em.reshape(2, -1)
                    e = e[:, :e.shape[1] // 2].cpu().numpy()
                    for a, b in zip(e[0].tolist(), e[1].tolist()):
                        nb[a].append(b)
                        nb[b].append(a)
            lists.append(nb)
        max_deg = max((len(x) for nb in lists for x in nb), default=0)
        width = max_deg + (0 if self.learn_eps else 1)
        m = sum(len(nb) for nb in lists)
        padded = np.full((m, max(width, 1)), -1, dtype=np.int64)
        first = np.full(m, -1, dtype=np.int64)
        row = 0
        for nb in lists:
            start = row
            for j, x in enumerate(nb):
                if x:
                    padded[row, :len(x)] = np.asarray(x, dtype=np.int64) + start
                    first[row] = x[0] + start
                if not self.learn_eps:
                    padded[row, max_deg] = start + j                    # graphcnn.py:73-75: the node itself, last
                    if not x and max_deg == 0:
                        first[row] = start + j
                row += 1
        return torch.from_numpy(padded), torch.from_numpy(first)

    def _max_neighbours(self, batch_graph):
        """Under max neighbour pooling, _padded_neighbours on the device: input gradients follow the reference's tie rule
        (the first entry of the padded list). (None, None) under the other poolings."""
        if self.neighbor_pooling_type != "max":
            return None, None
        padded, first = self._padded_neighbours(batch_graph)
        return padded.to(self.eps.device), first.to(self.eps.device)

    def _attribution_args(self, batch_graph, classes, what=None, counts=None, linear=False, occlusion=False):
        """The attribution methods' argument checks, in this order: eval() and `classes`; each of `counts` (name -> value)
        >= 1; no max neighbour pooling for a `linear` method; unless `what` is None (ROI saliency), BatchNorm running
        statistics and, for a non-empty batch and class list, one-hot features; for `occlusion` under max pooling a
        layer-0 max equal to its sum and no node without neighbours. `what` starts the messages. Returns (classes, counts
        as ints, out: float32 [B, len(classes), D] uninitialised, the host batch or None if there is nothing to compute)."""
        self.eval()
        classes = [int(c) for c in classes]
        n_cls = self.linears_prediction[0].weight.shape[0]
        if any(c < 0 or c >= n_cls for c in classes):
            raise ValueError("classes must lie in [0, %d), got %s" % (n_cls, classes))
        counts = {k: int(v) for k, v in (counts or {}).items()}
        if any(v < 1 for v in counts.values()):
            raise ValueError("%s must be >= 1, got %s" % (" and ".join(counts), " and ".join(map(str, counts.values()))))
        max_pool = self.neighbor_pooling_type == "max"
        if linear and max_pool:
            raise ValueError("%s sum or average neighbour pooling: max pooling is not linear in the input (use "
                             "compute_saliency_batched for its input gradient)" % what)
        if what is not None and not all(bn.track_running_stats for layer in range(self.num_layers)
                                        for _, bn in _engine.layer_units(self, layer)):
            raise ValueError("%s BatchNorm running statistics (eval mode per graph)" % what)
        d_in = _engine.layer_units(self, 0)[0][0].weight.shape[1]
        out = torch.empty(len(batch_graph), len(classes), d_in, dtype=torch.float32, device=self.eps.device)
        if len(batch_graph) == 0 or not classes:
            return classes, list(counts.values()), out, None
        h = self._host_batch(batch_graph)
        if what is not None and not h.onehot:
            raise ValueError("%s one-hot node features (util.py:114-116)" % what)
        if occlusion and max_pool and not h.max0_as_sum:
            raise ValueError("ROI occlusion under max neighbour pooling needs injective node tags and duplicate-free edge "
                             "lists in every graph (layer 0's max then equals its sum)")
        if occlusion and max_pool and h.has_isolated:
            raise ValueError("ROI occlusion under max neighbour pooling needs graphs without nodes without neighbours: "
                             "such a node pools the column minimum of the whole forward batch (graphcnn.py:137-143), so "
                             "its graph's occluded score would depend on the other copies in the pass")
        return classes, list(counts.values()), out, h

    def _layer0_base(self, rbs, params):
        """Layer 0 without its bias on the real batch `rbs` (one-hot): P = Agg(X) W1^T, from which a virtual batch's
        layer-0 output is written (engine.run_forward's z0). Returns (P, W1^T contiguous, eps or None, aggregation
        mode: 1 under average neighbour pooling, else 0)."""
        lin0 = _engine.layer_units(self, 0)[0][0]
        w1t = lin0.weight.detach().t().contiguous()
        mode = 1 if self.neighbor_pooling_type == "average" else 0
        eps_l = params[0][0:1] if self.learn_eps else None
        p0 = torch.empty(rbs.n_rows, lin0.weight.shape[0], dtype=torch.float32, device=self.eps.device)
        rbs.aggregate(w1t, rbs.tags, p0, mode, eps_l, None)
        return p0, w1t, eps_l, mode

    def _head_rows(self, classes):
        """d score_c / d g_f for each c in classes: the class-c rows of the prediction heads (graphcnn.py:228-231 in eval,
        no dropout)."""
        heads = [lin.weight.detach() for lin in self.linears_prediction]
        return [torch.cat([w[c] for w in heads]) for c in classes]

    def _virtual_forward(self, graphs, fill, params):
        """Eval forward of a virtual batch: `graphs` repeats graph objects of a real batch (the graph store resolves them
        to the same slots) and fill(vbs, bias, z) writes its layer-0 output. Returns (g_f, saved state)."""
        vbs = self._structure(graphs)
        g_f, _, sv = _engine.run_forward(self, vbs, None, False, False, None, params, _dist.SINGLE,
                                         z0=lambda bias, z: fill(vbs, bias, z))
        return g_f, sv

    def _class_scores(self, g_f, classes):
        """The eval class scores [V, len(classes)] of a virtual batch's g_f (no dropout in eval)."""
        return self._heads(g_f)[:, classes]

    def _heads(self, g_f):
        """graphcnn.py:228-231: sum over layers of dropout(Linear(pooled_h)). On the GPU: one libgnm launch forward, one
        backward (_HeadsFunction) instead of ~15 + ~25 small torch kernels whose launch latency sat on the critical path
        between the encoder's forward and backward graphs. The dropout masks are still drawn by L calls of F.dropout on
        [B, C] tensors - the same consumption of torch's generator, hence the same masks, as the reference's
        F.dropout(linear(pooled_h)) on that device."""
        n_cls = self.linears_prediction[0].weight.shape[0]
        if g_f.is_cuda and self.num_layers <= 16 and n_cls <= 8 and g_f.dtype == torch.float32:
            mask = None
            if self.training and self.final_dropout > 0.0:
                ones = torch.ones(g_f.shape[0], n_cls, dtype=torch.float32, device=g_f.device)
                mask = torch.stack([F.dropout(ones, self.final_dropout, training=True) for _ in range(self.num_layers)], 0)
            wb = [lin.weight for lin in self.linears_prediction] + [lin.bias for lin in self.linears_prediction]
            return _HeadsFunction.apply(g_f, mask, self.num_layers, *wb)
        f = self.hidden_dim
        score = 0
        for layer in range(self.num_layers):
            pooled_h = g_f[:, layer * f:(layer + 1) * f]
            score = score + F.dropout(self.linears_prediction[layer](pooled_h), self.final_dropout,
                                      training=self.training)
        return score

    # ---- reference API ------------------------------------------------------------------------
    def forward(self, batch_graph, latent=False):
        # data parallel applies to TRAINING forwards only. In eval mode BatchNorm uses the running statistics and no
        # exchange is needed, so a main.py-style test() on one rank (or with unequal chunk counts per rank) must not
        # enter a collective: the call is then single-process, each rank treating its list as the whole batch.
        comm = self._comm if self.training else _dist.SINGLE
        n_global = len(batch_graph) * comm.world
        rand_seq = np.random.permutation(n_global)          # graphcnn.py:199 (one numpy draw per call)
        h = self._host_batch(batch_graph)
        if h.uniform_n is None:
            # the reference's own DGI path needs equal-sized graphs (idx of graphcnn.py:198-201 and
            # the expand of discriminator.py:23-26 both assume M == B * N)
            raise RuntimeError("GIN_InfoMaxReg.forward needs graphs with the same number of nodes")
        plan = self._step_plan(h, n_global)
        if plan is not None:
            self._graph_store().h2d_bytes += plan.inputs.load(h, rand_seq)
            g_f, d_logit = _graphed.GraphedGINFunction.apply(plan, *_engine.flat_params(self))
        else:
            bs = self._structure(batch_graph, h)
            neg_idx = torch.from_numpy(rand_seq.astype(np.int32)).to(self.eps.device)
            runner = _engine.Runner(self, bs, neg_idx, self.training, True, comm)
            x = self._dense_features(batch_graph, bs)
            g_f, d_logit = _engine.GINFunction.apply(runner, x, *_engine.flat_params(self))
        c_logit = self._heads(g_f)
        if latent:
            return g_f.detach().cpu().numpy()
        return c_logit, d_logit

    def compute_saliency(self, batch_graph, cls):
        assert len(batch_graph) == 1
        return self.compute_saliency_batched(batch_graph, cls)

    def compute_saliency_batched(self, batch_graph, cls):
        """Gradient of the class-`cls` score wrt the (one-hot) input for a whole batch at once.
        Exact in eval mode: BatchNorm uses running statistics and Adj_block is block-diagonal,
        so each graph's rows equal its own `compute_saliency` result (graphcnn.py:254-299)."""
        self.eval()
        self.zero_grad()
        bs = self._structure(batch_graph)
        runner = _engine.Runner(self, bs, None, False, False, _dist.SINGLE, want_x_grad=True)
        runner.max_padded, runner.max_first = self._max_neighbours(batch_graph)
        x = self._dense_features(batch_graph, bs)
        if x is not None:
            x.requires_grad_()
        g_f, _ = _engine.GINFunction.apply(runner, x, *_engine.flat_params(self))
        score_over_layer = self._heads(g_f)
        predicting_class = torch.zeros([len(batch_graph), 2], device=g_f.device)     # graphcnn.py:263-264
        predicting_class[:, cls] = 1
        score_over_layer.backward(predicting_class)
        return runner.x_grad if x is None else x.grad

    def compute_roi_saliency_batched(self, batch_graph, classes):
        """ROI saliency: float32 [B, len(classes), D] device tensor whose entry [i, k] is
        `compute_saliency([batch_graph[i]], classes[k]).mean(0)` (up to fp32 rounding) - the node average that
        evaluate/plot_saliency_nii.py paints onto ROI volumes, without the [N, D] maps. One eval forward serves every
        class; each class then runs the hand-derived backward from the same saved state, and layer 0 reduces its
        gradient per graph instead of forming the map (engine.run_backward's ROI mode). Graphs may differ in size:
        each mean is over that graph's own nodes. Puts the model in eval() like compute_saliency but, unlike it, leaves
        every parameter's .grad untouched (no autograd pass runs)."""
        classes, _, out, h = self._attribution_args(batch_graph, classes)
        if h is None:
            return out
        bs = self._structure(batch_graph, h)
        max_padded, max_first = self._max_neighbours(batch_graph)
        x = self._dense_features(batch_graph, bs)
        params = [p.detach() for p in _engine.flat_params(self)]
        with torch.no_grad():
            _, _, sv = _engine.run_forward(self, bs, None, False, False, x, params, _dist.SINGLE, max_padded=max_padded)
            for k, row in enumerate(self._head_rows(classes)):
                dg_f = row.expand(len(batch_graph), -1).contiguous()
                _engine.run_backward(self, sv, params, dg_f, None, False, _dist.SINGLE, max_first=max_first, roi=out[:, k])
        return out

    def compute_integrated_gradients_batched(self, batch_graph, classes, steps=50, points_per_pass=1024,
                                             return_delta=False):
        """Integrated gradients with a zero baseline: float32 [B, len(classes), D] device tensor (and, with
        return_delta, the [B, len(classes)] completeness gap). Entry [i, k, d] is the node average over graph i of
        IG[n, d] = X[n, d] * (1/S) sum_s dF_c/dX(alpha_s X)[n, d], c = classes[k], alpha_s = (s + 1/2)/S (the midpoint
        rule, S = steps), F_c the eval-mode class score compute_saliency differentiates - the same node average as
        compute_roi_saliency_batched, so either can be painted onto ROIs; multiply by n_i for the per-graph sum.
        delta[i, k] = n_i * sum_d out[i, k, d] - (F_c(X_i) - F_c(0)) tends to 0 as steps grows (completeness).

        The path points run as one virtual batch per pass (exact in eval: a graph's outputs do not depend on its batch
        companions): one forward serves every class, one hand-derived backward per class follows, layer 0 runs once per
        real graph and no [N, D] tensor is formed (engine.run_forward's z0, run_backward's ig). A pass holds at most
        `points_per_pass` (graph, alpha) pairs: max(1, points_per_pass // steps) graphs, a graph's points spread over
        several passes when steps > points_per_pass. Graphs may differ in size. Puts the model in eval() and leaves
        every parameter's .grad untouched.

        Needs one-hot node features (util.py:114-116) and sum or average neighbour pooling: max pooling is not linear in
        the input, and its input gradient takes the [N, D] tie-rule route (compute_saliency_batched). ValueError
        otherwise, and for classes out of range or steps < 1."""
        classes, (steps, points_per_pass), out, h = self._attribution_args(
            batch_graph, classes, "integrated gradients need", dict(steps=steps, points_per_pass=points_per_pass),
            linear=True)
        dev = self.eps.device
        b, n_c = len(batch_graph), len(classes)
        delta = torch.empty(b, n_c, dtype=torch.float32, device=dev) if return_delta else None
        res = (out, delta) if return_delta else out
        if h is None:
            return res
        params = [p.detach() for p in _engine.flat_params(self)]
        dg_rows = self._head_rows(classes)
        alphas = ((torch.arange(steps, dtype=torch.float64) + 0.5) / steps).to(dev, torch.float32)
        per_chunk = max(1, points_per_pass // steps)
        points = min(steps, points_per_pass)
        with torch.no_grad():
            for i in range(0, b, per_chunk):
                chunk = batch_graph[i:i + per_chunk]
                rbs = self._structure(chunk)
                p0, w1t, eps_l, mode = self._layer0_base(rbs, params)          # z0(alpha) = alpha * p0 + b
                acc = torch.empty(n_c, rbs.n_rows, p0.shape[1], dtype=torch.float32, device=dev)
                for s0 in range(0, steps, points):
                    k = min(points, steps - s0)
                    fill = lambda vbs, bias, z: _ops.ig_expand(p0, bias, alphas[s0:s0 + k], rbs.node_off, k, z)
                    _, sv = self._virtual_forward([g for g in chunk for _ in range(k)], fill, params)
                    for j in range(n_c):
                        dg_f = dg_rows[j].expand(len(chunk) * k, -1).contiguous()
                        _engine.run_backward(self, sv, params, dg_f, None, False, _dist.SINGLE,
                                             ig=(acc[j], rbs.node_off, k, 1.0 / steps, s0 > 0))
                for j in range(n_c):
                    # IG = X o ((Agg^T acc) W1): per node the row dot with its tag's W1 column, averaged per ROI
                    t = torch.empty_like(p0)
                    rbs.aggregate(acc[j], None, t, 2 if mode == 1 else 0, eps_l, None)
                    _ops.ig_attribute(t, w1t, rbs.tags, rbs.node_off, out[i:i + len(chunk), j])
                if return_delta:
                    # F_c(X) - F_c(0): a forward-only virtual batch of the two endpoints
                    ends = torch.tensor([1.0, 0.0], dtype=torch.float32, device=dev)
                    fill = lambda vbs, bias, z: _ops.ig_expand(p0, bias, ends, rbs.node_off, 2, z)
                    g_f, _ = self._virtual_forward([g for g in chunk for _ in range(2)], fill, params)
                    score = self._class_scores(g_f, classes).view(len(chunk), 2, n_c)
                    n_g = torch.from_numpy(rbs.node_counts.astype(np.float32)).to(dev).unsqueeze(1)
                    delta[i:i + len(chunk)] = n_g * out[i:i + len(chunk)].sum(2) - (score[:, 0] - score[:, 1])
        return res

    def compute_roi_occlusion_batched(self, batch_graph, classes, occlusions_per_pass=1024):
        """ROI occlusion with a zero baseline: float32 [B, len(classes), D] device tensor whose entry [i, k, d] is
        (F_c(X_i) - F_c(X_i with column d set to 0)) / n_i, c = classes[k], F_c the eval-mode class score
        compute_saliency differentiates. The 1/n_i is the node-average convention of compute_roi_saliency_batched and
        compute_integrated_gradients_batched, so any of them can be painted onto ROIs; multiply by n_i for the score
        drop itself. Zeroing column d zeroes every node tagged d. A tag absent from graph i gives exactly 0.0 and costs
        no forward; a graph whose class score is not finite (average pooling's 0/0 at an isolated node under learn_eps)
        gives NaN for every ROI.

        The copies run as virtual batches of eval forwards (exact in eval: a graph's outputs do not depend on its batch
        companions). A pass holds, for each real graph in it, one baseline copy followed by occluded copies of that
        graph, so every difference is taken between two rows of the same forward; at most `occlusions_per_pass`
        virtual graphs in all, and at least one occluded copy. Layer 0 is aggregated once per call on the real batch
        and each copy's layer-0 output is that minus a rank-1 term (ops.occlusion_expand through engine.run_forward's
        z0); no [N, D] tensor is formed and no backward runs, so one forward serves every class. Graphs may differ in
        size. Puts the model in eval() and leaves every parameter's .grad untouched.

        Needs one-hot node features (util.py:114-116), BatchNorm running statistics, and under max neighbour pooling a
        batch whose layer-0 max equals its sum (injective tags and duplicate-free edge lists) and no node without
        neighbours (learn_eps: no self loop; max pooling gives such a node the column minimum of the whole forward batch,
        graphcnn.py:137-143, so a graph's score would depend on its companions). ValueError otherwise, and for classes
        out of range or occlusions_per_pass < 1."""
        classes, (occlusions_per_pass,), out, h = self._attribution_args(
            batch_graph, classes, "ROI occlusion needs", dict(occlusions_per_pass=occlusions_per_pass), occlusion=True)
        if h is None:
            return out
        out.zero_()                                                        # absent tags stay exactly 0
        dev = self.eps.device
        params = [p.detach() for p in _engine.flat_params(self)]
        cls_d = torch.tensor(classes, dtype=torch.int64, device=dev)
        inv_n = torch.from_numpy(1.0 / np.maximum(h.counts, 1)).to(dev, torch.float32)
        bad = torch.zeros(len(batch_graph), len(classes), dtype=torch.bool, device=dev)
        with torch.no_grad():
            rbs = self._structure(batch_graph, h)
            p0, w1t, eps_l, mode = self._layer0_base(rbs, params)          # a copy's z0: p0 + b minus a rank-1 term
            for v_graph, v_tag in occlusion_passes(h.node_off, rbs.tags.cpu().numpy(), occlusions_per_pass):
                v = len(v_graph)
                pos = np.arange(v, dtype=np.int32)
                base = np.maximum.accumulate(np.where(v_tag < 0, pos, 0)).astype(np.int32)
                copies = pos[v_tag >= 0]
                idx = torch.from_numpy(np.concatenate([v_graph, v_tag, copies, base[copies], pos[v_tag < 0]]))
                idx = idx.to(dev, non_blocking=True)
                vg_d, vt_d = idx[:v], idx[v:2 * v]
                n_k = len(copies)
                copy_d, base_d, bl_d = (t.long() for t in (idx[2 * v:2 * v + n_k], idx[2 * v + n_k:2 * v + 2 * n_k],
                                                           idx[2 * v + 2 * n_k:]))
                fill = lambda vbs, bias, z: _ops.occlusion_expand(p0, bias, w1t, rbs.rowptr, rbs.colidx, rbs.tags,
                                                                  rbs.node_off, rbs.n_max, vg_d, vt_d, vbs.node_off,
                                                                  mode, eps_l, z)
                g_f, _ = self._virtual_forward([batch_graph[g] for g in v_graph.tolist()], fill, params)
                score = self._class_scores(g_f, cls_d)                                # [V, C]
                g_k, d_k = vg_d[copy_d].long(), vt_d[copy_d].long()
                out[g_k, :, d_k] = (score[base_d] - score[copy_d]) * inv_n[g_k].unsqueeze(1)
                g_b = vg_d[bl_d].long()
                bad[g_b] = bad[g_b] | ~torch.isfinite(score[bl_d])
            out.masked_fill_(bad.unsqueeze(2), float("nan"))
        return out


def occlusion_passes(node_off, tags, occlusions_per_pass):
    """The virtual batches of compute_roi_occlusion_batched: a list of (v_graph, v_tag) int32 arrays, one per pass, graph
    major. For each real graph g (rows node_off[g] .. node_off[g+1] of `tags`) a pass holds one baseline copy (tag -1)
    followed by occluded copies of g, one per tag present in g in ascending order; a graph whose tags do not fit one pass
    continues in the next with a baseline copy of its own. A pass holds at most max(2, occlusions_per_pass) copies."""
    cap = max(2, int(occlusions_per_pass))
    passes, vg, vt = [], [], []
    for g in range(len(node_off) - 1):
        present = np.unique(tags[node_off[g]:node_off[g + 1]])
        i = 0
        while i < len(present):
            if len(vg) + 2 > cap:
                passes.append((vg, vt))
                vg, vt = [], []
            k = min(len(present) - i, cap - len(vg) - 1)
            vg.extend([g] * (k + 1))
            vt.append(-1)
            vt.extend(present[i:i + k].tolist())
            i += k
    if vg:
        passes.append((vg, vt))
    return [(np.asarray(a, dtype=np.int32), np.asarray(t, dtype=np.int32)) for a, t in passes]


GraphCNN = GIN_InfoMaxReg      # the name BASELINE.json's north_star uses for this class
