"""Host-side orchestration of the GIN + DGI hot path over the libgnm kernels.

What lives here (all of it replaces per-step Python/ATen work of the reference's
`GIN_InfoMaxReg.forward` / `compute_saliency`, models/graphcnn.py:194-299):

* `GraphStore`     - device-resident per-graph CSR cache (built once per `S2VGraph` by
                     `gnm_csr_build`), so a batch is assembled by offset arithmetic on the
                     device instead of re-running graphcnn.py:84-134 and shipping the sparse
                     index tensors H2D every step.
* `BatchStructure` - the block-diagonal CSR (`Adj_block`), node offsets (`graph_pool`) and
                     one-hot tags of one batch.
* `GINFunction`    - one `torch.autograd.Function` for the whole encoder + DGI scorer:
                     forward and a hand-derived backward, every M-sized tensor op is a
                     libgnm kernel. Only [B, L*F]-sized glue (sigmoid, u = c W^T, the
                     prediction heads) is left to torch.

The kernels are reached through `ops` (ctypes over the C ABI). There is no CPU path.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops as _ops
from . import dist as _dist


DENSE_MIN_DENSITY = 0.04      # use the tensor-core block kernel when nnz >= this fraction of sum N_g^2
FORCE_CSR_AGGREGATE = False    # test / A-B switch: always take the CSR gather kernel
FUSED_BWD_MAX = 64             # gnm_linear_bwd handles F_out, F_in <= 64; wider units take the unfused kernels
FORCE_UNFUSED_BACKWARD = False # test / A-B switch


def require_cuda(dev):
    if dev.type != "cuda":
        raise RuntimeError("GIN_InfoMaxReg runs on the libgnm CUDA kernels only (no CPU fallback): "
                           "call .to('cuda') first")


# ------------------------------------------------------------------------------------------
# graph store / batch structure
# ------------------------------------------------------------------------------------------

def _onehot_tags(feats, cache):
    """Return int32 tags if `feats` ([N, D] float) is exactly one-hot per row, else None."""
    key = (feats.data_ptr(), tuple(feats.shape), feats._version)
    if key in cache:
        return cache[key]
    tags = None
    if feats.dim() == 2 and feats.shape[1] > 0:
        f = feats.detach()
        if bool(((f == 0) | (f == 1)).all()) and bool((f.sum(1) == 1).all()):
            tags = f.argmax(1).to(torch.int32)
    cache[key] = tags
    return tags


class GraphStore(object):
    """Device cache of per-graph local CSRs, keyed on the identity of the caller's graph
    objects (the caller owns them and reuses them every step, main.py:26-28)."""

    def __init__(self, device, add_self_loops, max_bytes=None):
        """`max_bytes`: device-memory budget of the cache (default: a quarter of the device's memory). When a new
        chunk would exceed it the WHOLE store is dropped and the current batch re-built - callers that create fresh
        graph objects every step (augmentation, re-thresholding) therefore run at first-touch speed with bounded
        memory instead of leaking host and device memory. The key is the graph OBJECT: editing `graph.edge_mat` in
        place after its first use is not seen (call `GIN_InfoMaxReg.forget_graphs()` after such an edit)."""
        self.device = device
        self.add_self_loops = bool(add_self_loops)
        if max_bytes is None:
            max_bytes = torch.cuda.get_device_properties(device).total_memory // 4 if device.type == "cuda" else 1 << 62
        self.max_bytes = int(max_bytes)
        self.bytes = 0              # device bytes held by the stored CSRs / tags / bitmaps
        self.evictions = 0
        if hasattr(_ops, "prepare_device"):
            _ops.prepare_device(device)
        self.entries = {}           # id(graph) -> slot
        # slot table (one row per stored graph): rowptr / colidx / tag / bitmap addresses, n, nnz, onehot, isolated,
        # feature width, tag-sequence id. A batch is assembled from it with a handful of numpy gathers instead of per-graph Python.
        self._tab = np.zeros((0, 10), dtype=np.int64)
        self._n_slots = 0
        self._pins = []             # the graph objects (pins their ids) and the device buffers the addresses point into
        self._tag_cache = {}
        self._tag_seq_ids = {}      # bytes of an injective tag sequence -> small positive id (0 = not injective / not one-hot)
        self.h2d_bytes = 0          # bytes shipped host->device by the last ensure()/assemble()

    def _tag_seq_id(self, tags):
        """Graphs whose one-hot tags form the same injective sequence share an id (util.py:106-116 gives every subject
        one tag per ROI in the same ROI order); the layer-0 table gradient then is a plain sum over graphs."""
        if tags is None:
            return 0
        key = tags.numpy().tobytes()
        sid = self._tag_seq_ids.get(key)
        if sid is None:
            a = tags.numpy()
            sid = (len(self._tag_seq_ids) + 1) if np.unique(a).size == a.size else 0
            self._tag_seq_ids[key] = sid
        return sid

    def clear(self):
        self.entries.clear()
        self._tab = np.zeros((0, 10), dtype=np.int64)
        self._n_slots = 0
        self._pins = []
        self._tag_cache.clear()
        self.bytes = 0

    def _staging(self, e_total):
        """Pinned [2, E] int64 host buffer (grown geometrically, reused) for the edge lists of new graphs."""
        cap = getattr(self, "_stage_cap", 0)
        if cap < e_total or getattr(self, "_stage", None) is None:
            cap = max(e_total, int(cap * 1.5), 1)
            pin = self.device.type == "cuda"
            self._stage = torch.empty(2 * cap, dtype=torch.int64, pin_memory=pin)
            self._stage_cap = cap
        if self.device.type == "cuda":
            # the previous asynchronous copy out of this buffer must have finished before it is overwritten
            ev = getattr(self, "_stage_event", None)
            if ev is not None:
                ev.synchronize()
        return self._stage[:2 * e_total].view(2, e_total)

    def __len__(self):
        return len(self.entries)

    def ensure(self, graphs):
        new = []
        seen = set()
        for g in graphs:
            k = id(g)
            if k not in self.entries and k not in seen:
                seen.add(k)
                new.append(g)
        if not new:
            return
        if self.bytes > self.max_bytes and self.entries:
            # over budget: drop everything (buffers still referenced by enqueued kernels stay alive in torch's
            # stream-ordered allocator) and re-build this batch
            self.clear()
            self.evictions += 1
            return self.ensure(graphs)
        if any(getattr(g, "_edges_released", False) for g in new):
            raise RuntimeError("a graph whose edge list was released (synth.release_edges) is not in the store any more "
                               "(evicted: raise GraphStore.max_bytes) - it cannot be rebuilt")
        dev = self.device
        counts = [len(g.g) for g in new]
        ems = []
        for g, n in zip(new, counts):
            em = g.edge_mat
            if not torch.is_tensor(em):                 # an edgeless graph keeps util.py:17's `0`
                em = torch.zeros(2, 0, dtype=torch.int64)
            ems.append(em.reshape(2, -1).to(torch.int64))
        edge_counts = [int(e.shape[1]) for e in ems]
        edge_off = np.zeros(len(new) + 1, dtype=np.int64)
        np.cumsum(edge_counts, out=edge_off[1:])
        node_off = np.zeros(len(new) + 1, dtype=np.int64)
        np.cumsum(counts, out=node_off[1:])
        total_nodes = int(node_off[-1])
        # stage the edge lists once in pinned memory (no torch.cat temporary, no pageable bounce buffer) and ship
        # them with one asynchronous copy
        e_total = int(edge_off[-1])
        if dev.type == "cuda" and ems and all(e.is_cuda and e.device == dev for e in ems):
            # edge lists that already live on the device (synth.make_graphs_bulk(edges_on_device=True)): no host trip
            edges = edges_d = torch.cat(ems, 1) if len(ems) > 1 else ems[0].contiguous()
        else:
            edges = self._staging(e_total)
            for i, em in enumerate(ems):
                edges[:, int(edge_off[i]):int(edge_off[i + 1])].copy_(em)
            edges_d = edges.to(dev, non_blocking=True) if dev.type == "cuda" else edges.clone()
        edge_off_d = torch.from_numpy(edge_off).to(dev)
        node_off_d = torch.from_numpy(node_off.astype(np.int32)).to(dev)
        self.h2d_bytes += (0 if edges is edges_d and dev.type == "cuda" else edges.numel() * 8) + edge_off.nbytes + node_off.nbytes // 2
        if dev.type == "cuda":
            self._stage_event = torch.cuda.Event()
            self._stage_event.record()
        rowptr, colidx, status = _ops.csr_build(edges_d, edge_off_d, node_off_d, len(new), max(counts), total_nodes,
                                                self.add_self_loops, True)
        if int(status.item()) != 0:
            raise IndexError("edge_mat holds a node index outside [0, len(graph.g))")
        # one-hot tags of the node features (util.py:114-116), concatenated for the chunk
        tag_list, onehot, seq_ids = [], [], []
        for g in new:
            t = _onehot_tags(g.node_features, self._tag_cache)
            onehot.append(t is not None)
            seq_ids.append(self._tag_seq_id(t.cpu() if t is not None else None))
            tag_list.append(t if t is not None else torch.zeros(len(g.g), dtype=torch.int32))
        tags_d = torch.cat(tag_list).to(dev) if total_nodes > 0 else torch.zeros(0, dtype=torch.int32, device=dev)
        self.h2d_bytes += total_nodes * 4
        # adjacency bitmaps for the tensor-core aggregation (duplicate-free graphs only)
        words = np.array([n * ((n + 31) // 32) for n in counts], dtype=np.int64)
        bm_off = np.zeros(len(new) + 1, dtype=np.int64)
        np.cumsum(words, out=bm_off[1:])
        bm_off_d = torch.from_numpy(bm_off).to(dev)
        bitmap, dup = _ops.bitmap_build(rowptr, colidx, node_off_d, bm_off_d, len(new), int(bm_off[-1]))
        dup_h = dup.cpu().numpy()
        # graphs holding a node without any neighbour (average pooling gives 0/0 there, graphcnn.py:157-158)
        iso_h = np.zeros(len(new), dtype=bool)
        zero_rows = torch.nonzero((rowptr[1:] - rowptr[:-1]) == 0).flatten().cpu().numpy()
        if zero_rows.size:
            iso_h[np.searchsorted(node_off, zero_rows, side="right") - 1] = True
        self.h2d_bytes += bm_off.nbytes
        keep = (rowptr, colidx, tags_d, bitmap)
        self.bytes += sum(int(t.numel()) * t.element_size() for t in keep)
        rp0, ci0, tg0, bm0 = rowptr.data_ptr(), colidx.data_ptr(), tags_d.data_ptr(), bitmap.data_ptr()
        k = len(new)
        if self._n_slots + k > self._tab.shape[0]:
            grown = np.zeros((max(self._n_slots + k, 2 * self._tab.shape[0], 1024), 10), dtype=np.int64)
            grown[:self._n_slots] = self._tab[:self._n_slots]
            self._tab = grown
        t = self._tab[self._n_slots:self._n_slots + k]
        node_lo = np.asarray(node_off[:k], dtype=np.int64)
        nnz_base = np.asarray(edge_off[:k], dtype=np.int64) + (node_lo if self.add_self_loops else 0)
        t[:, 0] = rp0 + 4 * node_lo
        t[:, 1] = ci0 + 4 * nnz_base
        t[:, 2] = tg0 + 4 * node_lo
        t[:, 3] = np.where(np.asarray(dup_h[:k]) == 0, bm0 + 4 * np.asarray(bm_off[:k], dtype=np.int64), 0)
        t[:, 4] = counts
        t[:, 5] = np.asarray(edge_counts, dtype=np.int64) + (np.asarray(counts, dtype=np.int64) if self.add_self_loops else 0)
        t[:, 6] = np.asarray(onehot, dtype=np.int64)
        t[:, 7] = iso_h.astype(np.int64)
        t[:, 8] = [int(g.node_features.shape[1]) for g in new]
        t[:, 9] = seq_ids
        for i, g in enumerate(new):
            self.entries[id(g)] = self._n_slots + i
        self._n_slots += k
        self._pins.append((new, keep))

    def assemble_host(self, graphs):
        """Host half of batch assembly: per-slot addresses / offsets as numpy, plus batch-level flags."""
        b = len(graphs)
        getslot = self.entries.__getitem__
        try:
            idx = np.fromiter(map(getslot, map(id, graphs)), dtype=np.int64, count=b)
        except KeyError:
            self.ensure(graphs)
            idx = np.fromiter(map(getslot, map(id, graphs)), dtype=np.int64, count=b)
        t = self._tab[idx]                               # [b, 9]
        counts = np.ascontiguousarray(t[:, 4])
        packed = np.empty(5 * b + 1, dtype=np.int64)
        packed[0:b] = t[:, 0]
        packed[b:2 * b] = t[:, 1]
        packed[2 * b:3 * b] = t[:, 2]
        packed[3 * b] = 0
        np.cumsum(t[:, 5], out=packed[3 * b + 1:4 * b + 1])
        packed[4 * b + 1:5 * b + 1] = t[:, 3]
        node_off = np.zeros(b + 1, dtype=np.int32)
        np.cumsum(counts, out=node_off[1:])
        m, nnz = int(node_off[-1]), int(packed[4 * b])
        if nnz >= 2 ** 31:
            raise RuntimeError("batch adjacency has %d entries; int32 CSR holds < 2^31" % nnz)
        h = _HostBatch()
        h.b, h.m, h.nnz, h.packed, h.node_off, h.counts = b, m, nnz, packed, node_off, counts
        h.uniform_n = int(counts[0]) if b > 0 and bool((counts == counts[0]).all()) else None
        h.onehot = bool(t[:, 6].all())
        h.feat_dim = int(t[0, 8]) if b > 0 else 0
        h.n_max = int(counts.max()) if b > 0 else 0
        # tensor-core path: every graph has a bitmap (no duplicate edges) and the blocks are dense enough
        # that N^2 tensor-core MACs beat gathering nnz rows through L2 (break-even ~3-4 % density)
        has_bm = b > 0 and bool((t[:, 3] != 0).all())
        dense_enough = nnz >= DENSE_MIN_DENSITY * float((counts.astype(np.float64) ** 2).sum())
        h.dense = bool(has_bm and dense_enough)
        h.has_isolated = bool(t[:, 7].any())
        # every graph carries the same injective tag sequence (and so the same node count)
        h.same_tags = bool(b > 0 and t[0, 9] != 0 and (t[:, 9] == t[0, 9]).all() and h.uniform_n is not None)
        # max pooling of a one-hot layer-0 input is an OR of neighbour tags; when every graph's tags are injective and
        # its adjacency duplicate-free that OR equals the SUM aggregation, so layer 0 keeps the row-gather path
        h.max0_as_sum = bool(b > 0 and h.onehot and (t[:, 9] != 0).all() and has_bm)
        return h

    def assemble(self, h, graph_pooling_type, packed_d=None, node_off_d=None, nnz_capacity=None):
        """Device half: gather the stored CSRs of host batch `h` into the batch CSR (one kernel) and set the graph
        pooling's scale. `packed_d` / `node_off_d` are device copies of h.packed / h.node_off - a captured step passes
        its static buffers, with the batch CSR sized for `nnz_capacity` entries; by default they are copied here."""
        if packed_d is None:
            packed_d = torch.from_numpy(h.packed).to(self.device, non_blocking=True)
            node_off_d = torch.from_numpy(h.node_off).to(self.device, non_blocking=True)
            self.h2d_bytes += h.packed.nbytes + h.node_off.nbytes
        b = h.b
        nnz_cap = h.nnz if nnz_capacity is None else nnz_capacity
        # batches that run on the dense-block kernels never read the batch column indices: gather them lazily
        # (BatchStructure.colidx) - the copy is 2 x 195 MB of HBM traffic per step at B=1024, N=400
        lazy_cols = h.dense and not FORCE_CSR_AGGREGATE
        gather_args = (packed_d[0:b], packed_d[b:2 * b], None, node_off_d, packed_d[3 * b:4 * b + 1], b, h.m, nnz_cap)
        rowptr, colidx, tags = _ops.csr_batch_gather(packed_d[0:b], packed_d[b:2 * b], packed_d[2 * b:3 * b],
                                                     node_off_d, packed_d[3 * b:4 * b + 1], b, h.m, nnz_cap,
                                                     with_colidx=not lazy_cols)
        bs = BatchStructure()
        bs.n_graphs, bs.n_rows, bs.nnz = b, h.m, h.nnz
        bs.node_counts = h.counts
        bs.node_off = node_off_d
        bs.rowptr, bs._colidx, bs._gather_args = rowptr, colidx, gather_args
        bs.uniform_n = h.uniform_n
        bs.onehot = h.onehot
        bs.tags = tags if h.onehot else None
        bs.feat_dim = h.feat_dim
        bs.n_max = h.n_max
        bs.bitmap_addr = packed_d[4 * b + 1:5 * b + 1] if h.dense else None
        bs.has_isolated = h.has_isolated
        bs.same_tags = h.same_tags
        bs.max0_as_sum = h.max0_as_sum
        # graphcnn.py:118-120: 1 / len(graph.g) per graph under average pooling - from the device node offsets (no host
        # copy: this also runs under CUDA-graph capture)
        bs.pool_scale = (1.0 / (node_off_d[1:] - node_off_d[:-1]).to(torch.float32)
                         if graph_pooling_type == "average" else None)
        return bs


class _HostBatch(object):
    __slots__ = ("b", "m", "nnz", "packed", "node_off", "counts", "uniform_n", "onehot", "feat_dim", "n_max", "dense",
                 "has_isolated", "same_tags", "max0_as_sum")


class BatchStructure(object):
    """Adj_block (graphcnn.py:84-106) as int32 CSR + graph_pool (graphcnn.py:109-134) as node offsets."""

    __slots__ = ("n_graphs", "n_rows", "nnz", "node_counts", "node_off", "rowptr", "_colidx", "_gather_args",
                 "uniform_n", "onehot", "tags", "feat_dim", "pool_scale", "n_max", "bitmap_addr", "has_isolated",
                 "same_tags", "max0_as_sum")

    @property
    def colidx(self):
        """int32 global column ids of Adj_block; gathered on first use when the batch runs on the dense kernels."""
        if self._colidx is None:
            _, self._colidx, _ = _ops.csr_batch_gather(*self._gather_args)
        return self._colidx

    def _on_tc(self, src, dst, bias, mode):
        """Whether the batch runs on the tcgen05 dense-block kernel for these operands. Average pooling divides by the
        degree: an isolated node yields 0/0 = NaN in the reference, and a NaN row would poison its whole dense block
        (0 * NaN), so such batches keep the gather kernel."""
        return (self.bitmap_addr is not None and not FORCE_CSR_AGGREGATE and _ops.dense_aggregate_ok(src, dst, bias)
                and (mode == 0 or not self.has_isolated))

    def aggregate(self, src, src_map, dst, mode, eps, bias=None):
        """graphcnn.py:154-161 / :178-182 (and the transpose for backward): tensor-core dense-block kernel when
        the batch qualifies, CSR warp-per-row kernel otherwise."""
        if self._on_tc(src, dst, bias, mode):
            return _ops.aggregate_dense(self.bitmap_addr, self.node_off, self.rowptr, self.n_graphs, self.n_max,
                                        src, src_map, dst, mode, eps, bias)
        return _ops.aggregate(self.rowptr, self.colidx, src, src_map, dst, mode, eps, bias)

    def aggregate_bn(self, z, scale, shift, dst, pooled):
        """dst = Agg(relu(z*scale + shift)) (sum pooling, no self term) with the activated rows never written, and pooled
        (nullable) = their graph readout - the tcgen05 kernel's BatchNorm + ReLU on load. False, nothing launched, when
        the batch does not run on that kernel (the caller materialises h then)."""
        if not self._on_tc(z, dst, None, 0):
            return False
        return _ops.aggregate_dense(self.bitmap_addr, self.node_off, self.rowptr, self.n_graphs, self.n_max, z, None, dst,
                                    0, None, None, bn_scale=scale, bn_shift=shift, pooled=pooled,
                                    pool_scale=self.pool_scale)

    def aggregate_relu_bn_bwd(self, src, mode, eps, unit, d_pooled, d_score, u, d_neg, n_neg, dy, stats, tail=None):
        """Backward aggregation of `src` fused with the relu / BatchNorm backward reduction of `unit` (the last unit of
        the layer below) when the batch runs on the tcgen05 dense-block kernel; False, nothing launched, otherwise."""
        if FORCE_UNFUSED_BACKWARD or not self._on_tc(src, dy, None, mode):
            return False
        return _ops.aggregate_dense_relu_bn_bwd(self.bitmap_addr, self.node_off, self.rowptr, self.n_graphs, self.n_max,
                                                src, mode, eps, unit.z, unit.scale, unit.shift, unit.mean, unit.rstd,
                                                d_pooled, self.pool_scale, d_score, u, d_neg, n_neg, dy, stats, tail)

    def aggregate_table(self, table, dst, mode, eps, bias, stats, tail=None):
        """Layer 0 as a row gather of `table` when every graph carries the same tag sequence: dst = Agg(table[tags]) (+ self
        term) + bias and stats += its column statistics, the table staying resident in the kernel's shared memory
        (ops.aggregate_dense_table); False, nothing launched, when the batch does not run on the tcgen05 kernel."""
        if not (self.same_tags and self.uniform_n is not None and mode != 2 and self._on_tc(table, dst, bias, mode)):
            return False
        return _ops.aggregate_dense_table(self.bitmap_addr, self.node_off, self.rowptr, self.n_graphs, self.n_max, table,
                                          self.tags[:self.uniform_n], dst, mode, eps, bias, stats, tail)

    def aggregate_affine(self, dy, z, coef, dst, mode):
        """dst = Agg(coef[0]*dy + coef[1]*z + coef[2]) when the batch runs on the tcgen05 dense-block kernel (the affine
        is applied to the rows as they are loaded); False, with nothing launched, otherwise."""
        if not self._on_tc(dy, dst, None, mode):
            return False
        return _ops.aggregate_dense_affine(self.bitmap_addr, self.node_off, self.rowptr, self.n_graphs, self.n_max, dy, z,
                                           coef, dst, mode)


# ------------------------------------------------------------------------------------------
# parameter plumbing
# ------------------------------------------------------------------------------------------

def layer_units(model, layer):
    """The (Linear, BatchNorm1d) pairs of one GIN layer: mlp.py:27-38 + graphcnn.py:51."""
    mlp = model.mlps[layer]
    if mlp.linear_or_not:
        return [(mlp.linear, model.batch_norms[layer])]
    k = mlp.num_layers
    units = [(mlp.linears[j], mlp.batch_norms[j]) for j in range(k - 1)]
    units.append((mlp.linears[k - 1], model.batch_norms[layer]))
    return units


def flat_params(model):
    """The encoder / discriminator parameters in kernel order. The list of Parameter OBJECTS is cached on the model
    (walking the module tree costs ~0.1 ms and this runs several times per step on the host's critical path);
    `.to()` / `load_state_dict` keep the objects, assigning a new nn.Parameter to a submodule needs
    `model.release_graphs()` (which also drops this cache)."""
    ps = model.__dict__.get("_gnm_flat_params")
    if ps is None:
        ps = [model.eps, model.disc.f_k.weight, model.disc.f_k.bias]
        for layer in range(model.num_layers):
            for lin, bn in layer_units(model, layer):
                ps.extend([lin.weight, lin.bias, bn.weight, bn.bias])
        model.__dict__["_gnm_flat_params"] = ps
    return ps


def flat_buffers(model):
    """The BatchNorm buffers the kernels update in place (same set and order as `model.buffers()`, without walking the
    module tree: this runs every step to check that a captured CUDA graph still points at the live tensors)."""
    bns = model.__dict__.get("_gnm_flat_bns")
    if bns is None:
        bns = [bn for layer in range(model.num_layers) for _, bn in layer_units(model, layer)]
        model.__dict__["_gnm_flat_bns"] = bns
    # buffers are re-read every time: load_state_dict / .to() may replace the tensors. Read from the module's buffer
    # dict, as model.buffers() does: attribute access through nn.Module.__getattr__ costs 0.5 us per buffer
    return [t for bn in bns for t in bn._buffers.values() if t is not None]


class _Unit(object):
    """Saved forward state of one Linear->BatchNorm->ReLU unit."""
    __slots__ = ("w", "b", "gamma", "beta", "bn", "z", "scale", "shift", "mean", "rstd", "x_in", "count")


class _Saved(object):
    pass


# ------------------------------------------------------------------------------------------
# forward / backward
# ------------------------------------------------------------------------------------------

class _ZeroPool(object):
    """Zero-initialised accumulators (BatchNorm statistics, dW / db, scalar sums) handed out as 16-byte aligned views
    of a few large buffers: one fill kernel per buffer instead of one per accumulator (a training step has ~70)."""

    def __init__(self, dev, n_f32=1 << 15, n_f64=1 << 12):
        self.dev = dev
        self.cap = {torch.float32: n_f32, torch.float64: n_f64}
        self.buf = {torch.float32: None, torch.float64: None}
        self.used = {torch.float32: 0, torch.float64: 0}
        self.f64_chunks = []          # every float64 buffer handed out from (for batched post-processing)

    def _take(self, dtype, n):
        align = 4 if dtype == torch.float32 else 2
        n_al = (n + align - 1) // align * align
        if self.buf[dtype] is None or self.used[dtype] + n_al > self.buf[dtype].numel():
            self.buf[dtype] = torch.zeros(max(self.cap[dtype], n_al), dtype=dtype, device=self.dev)
            self.used[dtype] = 0
            if dtype == torch.float64:
                self.f64_chunks.append(self.buf[dtype])
        off = self.used[dtype]
        self.used[dtype] = off + n_al
        return self.buf[dtype], off

    def f32(self, *shape):
        n = 1
        for d in shape:
            n *= int(d)
        buf, off = self._take(torch.float32, n)
        return buf[off:off + n].view(*shape)

    def f64(self, n):
        """Returns (view, chunk index, offset) so that a caller can later address a converted copy of the chunk."""
        buf, off = self._take(torch.float64, int(n))
        return buf[off:off + int(n)], len(self.f64_chunks) - 1, off


FOLD_BN_TAILS = True           # A/B switch: BatchNorm finalisation in the last CTA of the kernel producing the statistics


def _bn_forward_tail(unit, stats, count, training, comm, buf=None):
    """Prepare the BatchNorm of `unit` (its Linear's output z is about to be produced together with `stats`): places
    scale / shift / mean / rstd in `buf` ([4, F], allocated when None) and returns the ops.BnTail the producer kernel may
    run in its last CTA - or None when this BatchNorm uses running statistics or the exchange needs NCCL.
    `_bn_affine(..., done=taken)` completes it."""
    dev = unit.z.device
    f = unit.z.shape[1]
    if buf is None:
        buf = torch.empty(4, f, dtype=torch.float32, device=dev)
    unit.scale, unit.shift, unit.mean, unit.rstd = buf[0], buf[1], buf[2], buf[3]
    bn = unit.bn
    use_batch = training or not bn.track_running_stats
    if not (FOLD_BN_TAILS and use_batch and hasattr(_ops, "BnTail")):
        return None
    p2p = comm.p2p_for(stats) if comm.world > 1 else None
    if comm.world > 1 and p2p is None:
        return None                   # the sums go through NCCL / gloo first
    track = bn.track_running_stats and training
    if track and bn.momentum is None:
        return None
    return _ops.BnTail(_ops.BnTail.FINALIZE, float(count * comm.world), unit.gamma, unit.mean, unit.rstd, beta=unit.beta,
                       eps=bn.eps, momentum=bn.momentum if track else 0.0, running_mean=bn.running_mean if track else None,
                       running_var=bn.running_var if track else None, nbt=bn.num_batches_tracked if track else None,
                       scale=unit.scale, shift=unit.shift, p2p=p2p)


def _bn_backward_tail(unit, stats, comm):
    """(coef, tail) for the BatchNorm backward of `unit`, whose [sum dy, sum dy*xhat] are about to be produced into `stats`:
    the producer kernel's last CTA all-reduces them (data parallel, peer memory) and writes gnm_bn_bwd_coeffs' output.
    (None, None) when this BatchNorm ran on running statistics or the exchange needs NCCL."""
    if not (FOLD_BN_TAILS and unit.count > 0.0 and hasattr(_ops, "BnTail")):
        return None, None
    p2p = comm.p2p_for(stats) if comm.world > 1 else None
    if comm.world > 1 and p2p is None:
        return None, None
    coef = torch.empty(3, unit.z.shape[1], dtype=torch.float32, device=unit.z.device)
    return coef, _ops.BnTail(_ops.BnTail.BWD_COEFFS, unit.count, unit.gamma, unit.mean, unit.rstd, coef=coef, p2p=p2p)


def _bn_affine(unit, stats, count, training, comm, done=False):
    dev = unit.z.device
    f = unit.z.shape[1]
    if getattr(unit, "scale", None) is None:
        buf = torch.empty(4, f, dtype=torch.float32, device=dev)
        unit.scale, unit.shift, unit.mean, unit.rstd = buf[0], buf[1], buf[2], buf[3]
    bn = unit.bn
    use_batch = training or not bn.track_running_stats
    if done:
        # the kernel that produced `stats` already ran gnm_bn_finalize's arithmetic in its last CTA
        unit.count = float(count * comm.world)
        return use_batch
    if use_batch:
        # data parallel: the global-batch sums. Over NVLink peer memory inside bn_finalize itself when the ranks share
        # a P2P communicator (dist.setup_p2p), else an NCCL / gloo all-reduce in front of it.
        p2p = comm.p2p_for(stats) if comm.world > 1 else None
        if comm.world > 1 and p2p is None:
            comm.all_reduce_sum(stats)
        unit.count = float(count * comm.world)
        track = bn.track_running_stats and training
        if track and bn.momentum is None:
            raise NotImplementedError("BatchNorm1d(momentum=None) is not used by the reference")
        _ops.bn_finalize(stats, unit.count, unit.gamma, unit.beta, bn.eps, bn.momentum if track else 0.0,
                         bn.running_mean if track else None, bn.running_var if track else None,
                         bn.num_batches_tracked if track else None, unit.scale, unit.shift, unit.mean, unit.rstd,
                         p2p=p2p)
    else:
        unit.count = 0.0
        _ops.bn_eval_affine(bn.running_mean, bn.running_var, unit.gamma, unit.beta, bn.eps, unit.scale, unit.shift,
                            unit.mean, unit.rstd)
    return use_batch


def first_argmax_from_padded(h, padded, cmin_values):
    """Arg-max of `torch.max(h_with_dummy[padded], dim=1)` (graphcnn.py:139-142) with the reference's tie rule - the FIRST
    entry of the padded neighbour list that attains the maximum - as source row ids ([M, F] int32, M = the dummy row).
    Structurally equivalent nodes (same closed neighbourhood) carry identical features, so exact ties at positive values
    do occur; parameter gradients do not care which of the tied nodes receives the gradient, the input gradient
    (saliency) does. `padded` [M, W] int64 with -1 pads; torch glue, used for the small batches of compute_saliency."""
    m = h.shape[0]
    hw = torch.cat([h, cmin_values.reshape(1, -1).to(h.dtype)], 0)
    idx = torch.where(padded >= 0, padded, torch.full_like(padded, m))
    vals = hw[idx]                                                   # [M, W, F]
    best = vals.max(1, keepdim=True)[0]
    at_max = vals == best
    first = at_max & (at_max.to(torch.int32).cumsum(1) == 1)         # exactly one True per (row, feature)
    pos = first.to(torch.float32).argmax(1)                          # [M, F]
    return idx.gather(1, pos).to(torch.int32)


BN_ON_LOAD = True              # A/B switch: layers' h formed on load from z by its consumers instead of materialised


def _materialise_plan(model, bs, with_dgi):
    """Which layers' h = relu(BN(z)) must be written to memory ([L] bools), and whether the DGI kernels read z with the
    BatchNorm on load. A layer's h is materialised only when one of its consumers cannot form it on load: the next
    layer's aggregation off the tcgen05 single-pass kernel (CSR, mma.sync, more than TC_MAX_NODES nodes, max / average
    pooling, the eps self term, F > 64), learn_eps (the backward's d eps reads h), or a DGI shape off the 64-wide kernels."""
    L, F = model.num_layers, model.hidden_dim
    on_load = BN_ON_LOAD and getattr(_ops, "BN_ON_LOAD", False)
    agg_ok = (on_load and not FORCE_CSR_AGGREGATE and bs.bitmap_addr is not None and bs.n_max <= _ops.TC_MAX_NODES and
              _ops.DENSE_IMPL[0] != 1 and model.neighbor_pooling_type == "sum" and not model.learn_eps and
              F % 4 == 0 and F <= 64)
    dgi_ok = on_load and F == 64 and L <= 5
    need = [not agg_ok if layer < L - 1 else False for layer in range(L)]
    if with_dgi and not dgi_ok:
        need = [True] * L
    return need, on_load and with_dgi and dgi_ok


def run_forward(model, bs, neg_idx, training, with_dgi, x_dense, params, comm, max_padded=None, bce=None, z0=None):
    """graphcnn.py:194-251 (and :254-294 when with_dgi is False). Returns (g_f, d_logit, saved).
    z0 = fill(bias, z), eval only: `bs` is a virtual batch whose graphs repeat those of a real batch, and fill writes
    layer 0's first Linear output z [M, F] (bias included) from the real batch's aggregation p = Agg(X) W1^T - no
    aggregation runs on the virtual batch at layer 0. Integrated gradients: alpha[s] * p + bias at every path point
    (ops.ig_expand); occlusion: p + bias minus the rank-1 term of the occluded column (ops.occlusion_expand).
    bce = (grad_scale, loss_scale, loss_acc): the caller's loss on d_logit is BCEWithLogits against main.py:32's targets
    with these scales (driver.Trainer). The scoring pass then also adds the loss to loss_acc and forms the scorer's
    backward (saved.scored = (d_score, du, s2, d_bias)) when its kernel takes the shape; saved.scored is None otherwise
    and the caller applies the loss to d_logit itself."""
    dev = params[0].device
    L, F = model.num_layers, model.hidden_dim
    M, B = bs.n_rows, bs.n_graphs
    learn_eps = model.learn_eps
    average = model.neighbor_pooling_type == "average"
    eps_p, disc_w, disc_b = params[0], params[1], params[2]
    it = iter(params[3:])
    sv = _Saved()
    sv.layers = []
    sv.bs = bs
    sv.training = training
    sv.with_dgi = with_dgi
    sv.x_dense = x_dense
    sv.scored = None
    sv.F = F
    # Each layer's h = relu(BN(z_last)) is read on load from its last unit's z (z_all[layer]) with that unit's scale /
    # shift (bn_all[layer, :2]) by the next layer's aggregation - which also forms the layer's readout - and by the DGI
    # kernels; h_all exists only when some layer's h has a consumer that cannot do that (_materialise_plan).
    need_h, dgi_on_load = _materialise_plan(model, bs, with_dgi)
    h_all = torch.empty(L, M, F, dtype=torch.float32, device=dev) if any(need_h) else None
    z_all = torch.empty(L, M, F, dtype=torch.float32, device=dev) if not all(need_h) else None
    bn_all = torch.empty(L, 4, F, dtype=torch.float32, device=dev) if z_all is not None else None
    g_f = torch.empty(B, L * F, dtype=torch.float32, device=dev)
    sv.h_all = h_all
    use_gather0 = x_dense is None
    if use_gather0 and not bs.onehot:
        raise RuntimeError("internal: gather path needs one-hot node features")
    maxpool = model.neighbor_pooling_type == "max"
    if maxpool and use_gather0 and not bs.max0_as_sum:
        raise RuntimeError("internal: max pooling keeps the layer-0 gather only for injective tags on duplicate-free graphs")
    sv.use_gather0 = use_gather0
    sv.max_state = {}          # layer -> (argmax [M, F_in] int32, packed column minimum) under max pooling
    sv.batch_stats = []
    zp = _ZeroPool(dev)
    for layer in range(L):
        units = []
        for lin, bn in layer_units(model, layer):
            u = _Unit()
            u.w, u.b, u.gamma, u.beta = next(it), next(it), next(it), next(it)
            u.bn = bn
            units.append(u)
        eps_l = eps_p[layer:layer + 1] if learn_eps else None
        h_prev = h_all[layer - 1] if layer > 0 and need_h[layer - 1] else None
        pooled = None
        for j, u in enumerate(units):
            n_out = u.w.shape[0]
            last_unit = j == len(units) - 1 and z_all is not None
            u.z = z_all[layer] if last_unit else torch.empty(M, n_out, dtype=torch.float32, device=dev)
            u.scale = None
            stats = zp.f64(2 * n_out)[0]
            tail = _bn_forward_tail(u, stats, M, training, comm, buf=bn_all[layer] if last_unit else None)
            done = False
            if j == 0:
                if layer == 0 and use_gather0 and z0 is not None:
                    # z0 from one real-batch aggregation (eval: the BatchNorm reads no statistics of z0)
                    z0(u.b, u.z)
                    u.x_in = None
                elif layer == 0 and use_gather0:
                    # first layer as a row gather of W1^T (X_concat is one-hot): no dense X, no GEMM
                    w1t = u.w.detach().t().contiguous()
                    sv.w1t = w1t
                    done = tail is not None and bs.aggregate_table(w1t, u.z, 1 if average else 0, eps_l, u.b, stats, tail)
                    if not done and not bs.aggregate_table(w1t, u.z, 1 if average else 0, eps_l, u.b, stats):
                        bs.aggregate(w1t, bs.tags, u.z, 1 if average else 0, eps_l, u.b)
                        _ops.col_stats(u.z, stats)
                    u.x_in = None
                elif layer > 0 and h_prev is None:
                    # h of the layer below formed on load from its z, and that layer's readout formed with it
                    below = sv.layers[layer - 1][-1]
                    pooled = torch.empty(M, F, dtype=torch.float32, device=dev)
                    g_below = g_f[:, (layer - 1) * F:layer * F]
                    if not bs.aggregate_bn(below.z, below.scale, below.shift, pooled, g_below):
                        h_tmp = torch.empty(M, F, dtype=torch.float32, device=dev)
                        _ops.bn_relu_readout(below.z, below.scale, below.shift, h_tmp, bs.node_off, B, bs.pool_scale,
                                             g_below)
                        bs.aggregate(h_tmp, None, pooled, 0, None, None)
                    done = bool(_ops.linear(pooled, u.w, False, u.b, None, None, u.z, stats, tail))
                    u.x_in = pooled
                else:
                    src = x_dense if layer == 0 else h_prev
                    pooled = torch.empty(M, src.shape[1], dtype=torch.float32, device=dev)
                    if maxpool:
                        # graphcnn.py:137-143: max over the padded neighbour list, dummy row = column minimum of h
                        cmin = _ops.col_min(src)
                        amax = torch.empty(M, src.shape[1], dtype=torch.int32, device=dev)
                        _ops.aggregate_max(bs.rowptr, bs.colidx, src, cmin, eps_l, pooled, amax)
                        if max_padded is not None:
                            # an input gradient is wanted: ties must go where torch.max sends them (list order)
                            amax = first_argmax_from_padded(src, max_padded, _ops.col_min_values(cmin)).contiguous()
                        sv.max_state[layer] = (amax, cmin)
                    else:
                        bs.aggregate(src, None, pooled, 1 if average else 0, eps_l, None)
                    done = bool(_ops.linear(pooled, u.w, False, u.b, None, None, u.z, stats, tail))
                    u.x_in = pooled
            else:
                p = units[j - 1]
                done = bool(_ops.linear(p.z, u.w, False, u.b, p.scale, p.shift, u.z, stats, tail))
                u.x_in = None          # recomputed from p.z with p's affine + ReLU
            _bn_affine(u, stats, M, training, comm, done=done)
        last = units[-1]
        if need_h[layer] or layer == L - 1:
            # the readout (writing h only where a consumer needs it); the other layers' readouts come with the next
            # layer's aggregation
            _ops.bn_relu_readout(last.z, last.scale, last.shift, h_all[layer] if need_h[layer] else None, bs.node_off, B,
                                 bs.pool_scale, g_f[:, layer * F:(layer + 1) * F])
        sv.layers.append(units)
    # what the DGI kernels read: the pre-BatchNorm z with scale | shift applied on load, or the materialised h
    nf, nf_bn = (z_all, bn_all[:, :2]) if dgi_on_load else (h_all, None)
    sv.nf, sv.nf_bn = nf, nf_bn
    bn_kw = {"bn": nf_bn} if nf_bn is not None else {}
    d_logit = None
    if with_dgi:
        # discriminator.py:19-38 refactored: sc = <h, u_g> + b with u_g = W c_g (c = sigmoid(g_f), graphcnn.py:238-239)
        # c = sigmoid(g_f) and u = c W^T in one launch (W = disc.f_k.weight[0], [L*F, L*F] row-major: u[b,i] = sum_j c[b,j] W[i,j])
        lf = L * F
        c = torch.empty(B, lf, dtype=torch.float32, device=dev)
        u_mat = torch.empty(B, lf, dtype=torch.float32, device=dev)
        w_d = disc_w[0]
        _ops.small_gemm(g_f, (g_f.stride(0), 1), w_d, (1, w_d.stride(0)), u_mat, B, lf, lf, sigmoid_a_out=c)
        b_neg = neg_idx.shape[0]
        sv.rows_region = None
        if comm.world > 1:
            # the negatives only ever read global rows [0, B_global) of n_f: rank 0 owns them
            my_neg = neg_idx[comm.rank * B:(comm.rank + 1) * B].contiguous()
            reg = comm.region("dgi_rows", 2 * b_neg * lf * 4)
            if reg is not None:
                # over NVLink peer memory: rank 0 gathers the rows into ITS region, a barrier, and every rank's score
                # kernels read the B rows their permutation slice names straight from rank 0's memory (1.3 MB per rank
                # at B = 1024 instead of a broadcast of the whole [B_global, L*F] table)
                neg_table = reg.tensor(0, 0, (b_neg, lf))
                if comm.rank == 0:
                    _ops.gather_nf_rows(nf, b_neg, out=neg_table, **bn_kw)
                comm.p2p_barrier()
                sv.rows_region = reg
            else:
                neg_table = _ops.gather_nf_rows(nf, b_neg, **bn_kw) if comm.rank == 0 else \
                    torch.empty(b_neg, lf, dtype=torch.float32, device=dev)
                comm.broadcast(neg_table, 0)
        else:
            neg_table = _ops.gather_nf_rows(nf, b_neg, **bn_kw)
            my_neg = neg_idx
        d_logit = torch.empty(2 * M, 1, dtype=torch.float32, device=dev)
        scored = False
        if bce is not None:
            # the BCE gradient of a score is local: one pass over n_f forms the scores, the loss and the scorer's
            # backward (dgi_score_bwd would read the same L slices again)
            d_score = torch.empty(M, dtype=torch.float32, device=dev)
            du = torch.empty(B, lf, dtype=torch.float32, device=dev)
            s2 = torch.empty(B, dtype=torch.float32, device=dev)
            d_bias = zp.f64(1)[0]
            scored = _ops.dgi_score_train(nf, u_mat, neg_table, my_neg, bs.node_off, B, disc_b, bce[0], bce[1],
                                          d_logit, d_score, du, s2, d_bias, bce[2], **bn_kw)
            if scored:
                sv.scored = (d_score, du, s2, d_bias)
        if not scored:
            _ops.dgi_score_fwd(nf, u_mat, neg_table, my_neg, bs.node_off, B, disc_b, d_logit, **bn_kw)
        sv.c, sv.u_mat, sv.neg_table, sv.my_neg, sv.neg_idx = c, u_mat, neg_table, my_neg, neg_idx
    return g_f, d_logit, sv


def max_pool_onehot_input_grad(bs, p, first, eps):
    """Gradient of `maxpool(X) [+ (1 + eps) X]` (graphcnn.py:137-143 on the one-hot layer-0 input) wrt X, given
    p = d loss / d pooled [M, D]. torch.max sends the gradient of entry (i, d) to ONE member of node i's padded
    neighbour list: the member whose tag is d (value 1, unique for injective tags) if there is one, else - every
    candidate ties at 0 - the FIRST entry of the list (`first[i]`, the reference's neighbour order; -1 = the list
    holds pads only, the gradient then lands on the row that supplied the dummy row's minimum). [B, L*F]-style glue in
    torch (saliency runs one graph, or a few, per call)."""
    m, d = p.shape
    dev = p.device
    tags = bs.tags.long()
    rp, ci = bs.rowptr.long(), bs.colidx.long()
    rows = torch.repeat_interleave(torch.arange(m, device=dev), rp[1:] - rp[:-1])
    hit_cols = tags[ci]                                              # list member ci holds a 1 in column tags[ci]
    d_x = torch.zeros(m, d, dtype=p.dtype, device=dev)
    d_x.index_put_((ci, hit_cols), p[rows, hit_cols], accumulate=True)
    has_one = torch.zeros(m, d, dtype=torch.bool, device=dev)
    has_one[rows, hit_cols] = True
    rest = p.masked_fill(has_one, 0.0)                               # columns in which every candidate is 0
    ok = first >= 0
    d_x.index_add_(0, first[ok], rest[ok])
    if bool((~ok).any()):
        cols = torch.arange(d, device=dev)
        r_min = torch.where(tags[0] == cols, 1, 0)                   # first row whose entry in column d is the minimum 0
        d_x.index_put_((r_min, cols), rest[~ok].sum(0), accumulate=True)
    if eps is not None:
        d_x += (1.0 + eps) * p
    return d_x


def run_backward(model, sv, params, dg_f, dd_logit, need_x_grad, comm, max_first=None, roi=None, ig=None):
    """Hand-derived backward of `run_forward`. Returns (dX or None, [grad per flat param]).
    roi ([B, D] view, nullable): ROI mode - roi[g] receives the node average of graph g's input gradient,
    (1/n_g) sum_{n in g} dX[n], formed without dX where the layer-0 aggregation is linear (ops.segment_weighted_colsum:
    mean_n (Agg^T dz)[n] = (1/n_g) sum_m w_m dz[m], w_m the operator's row sums). Layer 0's parameter gradients are not
    formed then. Nothing here writes the saved forward state, so one forward serves a backward per class.
    ig = (acc, node_off, points, weight, accumulate), for a forward whose z0 ran ops.ig_expand: integrated-gradients
    mode - the layer-0 dz of every path point, weighted, is summed onto the real rows acc [M_real, F] (ops.ig_accumulate;
    written, or added to when accumulate). Agg^T and W1 are applied once per real batch by the caller. Layer 0's parameter
    gradients are not formed."""
    bs = sv.bs
    dev = params[0].device
    L = model.num_layers
    M, B = bs.n_rows, bs.n_graphs
    F = sv.F
    learn_eps = model.learn_eps
    average = model.neighbor_pooling_type == "average"
    bwd_mode = 2 if average else 0
    eps_p, disc_w, disc_b = params[0], params[1], params[2]
    grads = [None] * len(params)
    zp = _ZeroPool(dev)
    from_f64 = []         # (grad index, chunk, offset, length, scaled): float64 accumulators converted in one go at the end
    d_eps = None
    if learn_eps:
        d_eps, c_, o_ = zp.f64(L)
        from_f64.append((0, c_, o_, L, False))

    d_pooled = dg_f
    d_score = u_mat = d_neg = None
    n_neg = 0
    if sv.with_dgi and (dd_logit is not None or sv.scored is not None):
        if sv.scored is not None:
            d_score, du, s2, d_bias = sv.scored            # formed by run_forward's scoring pass
            grads[2] = d_bias.to(torch.float32).view(tuple(params[2].shape))
        else:
            dd = dd_logit.contiguous().view(-1)
            d_score = dd[:M]
            du = torch.empty(B, L * F, dtype=torch.float32, device=dev)
            s2 = torch.empty(B, dtype=torch.float32, device=dev)
            d_bias, c_, o_ = zp.f64(1)
            from_f64.append((2, c_, o_, 1, False))
            bn_kw = {"bn": sv.nf_bn} if sv.nf_bn is not None else {}
            _ops.dgi_score_bwd(sv.nf, dd, sv.neg_table, sv.my_neg, bs.node_off, B, du, s2, d_bias, **bn_kw)
        # [B, L*F]-sized glue of u = c W^T, c = sigmoid(g_f): dW[i,j] = sum_b du[b,i] c[b,j];
        # d g_f = dg_f (heads) + (du W) c (1 - c); gradient reaching the shuffled rows n_f[perm[g]]
        lf = L * F
        w_d = disc_w[0]
        d_w = torch.empty(1, lf, lf, dtype=torch.float32, device=dev)
        _ops.small_gemm(du, (1, du.stride(0)), sv.c, (sv.c.stride(0), 1), d_w[0], lf, lf, B)
        grads[1] = d_w
        dgs = torch.empty(B, lf, dtype=torch.float32, device=dev)
        dg_heads = d_pooled.contiguous() if d_pooled is not None else None
        _ops.small_gemm(du, (du.stride(0), 1), w_d, (w_d.stride(0), 1), dgs, B, lf, lf, dsig_s=sv.c, dsig_add=dg_heads)
        d_pooled = dgs
        n_neg = sv.neg_idx.shape[0]
        if comm.world > 1 and sv.rows_region is not None:
            # every global row j < B_global is named by exactly one (rank, graph) - the indices are a permutation -
            # so the gradient of the shuffled rows is a pure scatter: each rank writes ITS rows into rank 0's region
            # (remote stores over NVLink), a barrier, and rank 0 reads the complete [B_global, L*F] block
            d_neg = sv.rows_region.tensor(0, n_neg * lf * 4, (n_neg, lf))
            _ops.scatter_scaled_rows(sv.my_neg, s2, sv.u_mat, d_neg)
            comm.p2p_barrier()
            if comm.rank != 0:
                d_neg, n_neg = None, 0
        else:
            d_neg = torch.empty(n_neg, lf, dtype=torch.float32, device=dev)
            _ops.dgi_neg_grad(sv.my_neg, s2, sv.u_mat, d_neg)
            if comm.world > 1:
                comm.reduce_sum(d_neg, 0)
                if comm.rank != 0:
                    d_neg, n_neg = None, 0
        u_mat = sv.u_mat
    if d_pooled is None:
        d_pooled = torch.zeros(B, L * F, dtype=torch.float32, device=dev)
    d_pooled = d_pooled.contiguous()

    d_h = None        # gradient reaching h_all[layer] from layer+1's aggregation
    ready = None      # (dy, stats, coef) of the next unit when the kernel that ran the unit above already produced them
    d_x = None
    # per layer: the slices of the readout gradient and of the DGI terms that reach its h directly
    side = [(d_pooled[:, s], u_mat[:, s] if u_mat is not None else None, d_neg[:, s] if d_neg is not None else None)
            for s in (slice(layer * F, (layer + 1) * F) for layer in range(L))]

    def agg_transpose(layer, dp, eps_l):
        """Agg^T dp for the aggregation that feeds `layer` (its max-pooling backward when that layer ran max pooling)."""
        out = torch.empty(M, dp.shape[1], dtype=torch.float32, device=dev)
        if layer in sv.max_state:
            amax, cmin = sv.max_state[layer]
            _ops.aggregate_max_bwd(bs.rowptr, bs.colidx, dp, amax, cmin, eps_l, out)
        else:
            bs.aggregate(dp, None, out, bwd_mode, eps_l, None)
        return out

    def bn_coef(u, stats, coef_ready, p2p=None):
        """[3, F] BatchNorm-backward coefficients of `u`, dz = A*dy + B*z + C: coef_ready when the kernel that produced
        `stats` already formed them in its last CTA."""
        if coef_ready is not None:
            return coef_ready
        coef = torch.empty(3, u.w.shape[0], dtype=torch.float32, device=dev)
        _ops.bn_bwd_coeffs(stats if u.count > 0.0 else None, u.count, u.gamma, u.mean, u.rstd, coef, p2p=p2p)
        return coef

    def max_pool_x_grad(dz, w, eps_l):
        """Input gradient of the one-hot layer 0 under max pooling, from dz = d loss / d z_0."""
        if max_first is None:
            raise RuntimeError("input gradients under max pooling need the neighbour-list order "
                               "(use compute_saliency / compute_saliency_batched)")
        dp0 = torch.empty(M, w.shape[1], dtype=torch.float32, device=dev)
        _ops.linear(dz, w, True, None, None, None, dp0, None)         # d loss / d pooled_0 = dz @ W1
        return max_pool_onehot_input_grad(bs, dp0, max_first, eps_l)

    def through_aggregation(layer, dp, eps_l):
        """dp = d loss / d pooled_layer, the output of the layer's neighbour aggregation: d eps, then the gradient of the
        aggregation's input. Above layer 0 that sets d_h of the layer below = Agg^T dp - or, when the aggregation kernel
        also ran that layer's relu / BatchNorm backward reduction, `ready`. At layer 0 it forms the ROI reduction or d_x."""
        nonlocal d_h, ready, d_x
        roi0 = layer == 0 and roi is not None
        if learn_eps and not roi0:
            _ops.dot_rows(dp, sv.x_dense if layer == 0 else sv.h_all[layer - 1], None, d_eps[layer:layer + 1])
        if layer > 0:
            below = sv.layers[layer - 1][-1]
            if layer not in sv.max_state and below.z.shape[1] == dp.shape[1]:
                dy_b = torch.empty(M, dp.shape[1], dtype=torch.float32, device=dev)
                st_b = zp.f64(2 * dp.shape[1])
                coef_b, tail_b = _bn_backward_tail(below, st_b[0], comm)
                d_pool_b, u_b, d_neg_b = side[layer - 1]
                if bs.aggregate_relu_bn_bwd(dp, bwd_mode, eps_l, below, d_pool_b, d_score, u_b, d_neg_b, n_neg, dy_b,
                                            st_b[0], tail_b):
                    d_h, ready = None, (dy_b, st_b, coef_b)
                    return
            d_h = agg_transpose(layer, dp, eps_l)
        elif roi0:
            # the node average of d_x = Agg^T dp: the reduction of dp itself with the operator's row sums; under max
            # pooling, which is not linear, of d_x - the [M, D] route
            if 0 in sv.max_state:
                _ops.segment_weighted_colsum(agg_transpose(0, dp, eps_l), bs.node_off, roi)
            else:
                _ops.segment_weighted_colsum(dp, bs.node_off, roi, rowptr=bs.rowptr, mode=1 if average else 0, eps=eps_l)
        elif need_x_grad:
            d_x = agg_transpose(0, dp, eps_l)

    pidx = 3 + 4 * sum(len(u) for u in sv.layers)
    for layer in range(L - 1, -1, -1):
        units = sv.layers[layer]
        pidx -= 4 * len(units)
        eps_l = eps_p[layer:layer + 1] if learn_eps else None
        need_dp = layer > 0 or need_x_grad or learn_eps or roi is not None      # d loss / d pooled_layer has a use
        dz = None
        for j in range(len(units) - 1, -1, -1):
            u = units[j]
            n_out, n_in = u.w.shape[0], u.w.shape[1]
            if ready is not None:
                (dy, (stats, st_chunk, st_off), coef_ready), ready = ready, None
            else:
                dy = torch.empty(M, n_out, dtype=torch.float32, device=dev)
                stats, st_chunk, st_off = zp.f64(2 * n_out)
                coef_t, tail_t = _bn_backward_tail(u, stats, comm)
                if j == len(units) - 1:
                    d_pool_l, u_l, d_neg_l = side[layer]
                    d_out = (d_h, d_pool_l, bs.pool_scale, d_score, u_l, d_neg_l, n_neg)
                else:
                    d_out = (dz, None, None, None, None, None, 0)
                took = _ops.relu_bn_bwd_reduce(u.z, u.scale, u.shift, u.mean, u.rstd, *d_out, bs.node_off, B, dy, stats,
                                               tail=tail_t)
                coef_ready = coef_t if took is True else None
            use_batch = u.count > 0.0
            gather0 = j == 0 and layer == 0 and sv.use_gather0
            fused = (not gather0) and (not FORCE_UNFUSED_BACKWARD) and n_out <= FUSED_BWD_MAX and n_in <= FUSED_BWD_MAX
            p2p = None
            if use_batch and comm.world > 1 and coef_ready is None:
                # global-batch [sum dy, sum dy*xhat]: exchanged inside bn_bwd_coeffs (fused path) or by the small
                # peer-memory all-reduce kernel when the ranks share a P2P communicator, else NCCL / gloo (a tail has
                # already done the exchange, in place, when coef_ready is set)
                p2p = comm.p2p_for(stats)
                if p2p is None:
                    comm.all_reduce_sum(stats)
                elif not fused:
                    p2p.allreduce(stats)
                    p2p = None
            gi = pidx + 4 * j
            # d beta = sum dy, d gamma = sum dy * xhat (converted, and scaled to this rank's share, at the end)
            scaled = use_batch and comm.world > 1
            from_f64.append((gi + 3, st_chunk, st_off, n_out, scaled))
            from_f64.append((gi + 2, st_chunk, st_off + n_out, n_out, scaled))
            dw = zp.f32(*u.w.shape)
            db = zp.f32(*u.b.shape)
            if gather0 and ig is not None:
                # integrated gradients: sum_s w * dz_s = w * cA o sum_s dy_s (eval: cB = cC = 0) on the real rows - Agg^T
                # and W1 are linear, so they need not run per path point
                acc, real_off, points, weight, accumulate = ig
                _ops.ig_accumulate(dy, bn_coef(u, stats, coef_ready), real_off, points, weight, acc, accumulate)
                continue
            if gather0 and roi is not None:
                # ROI mode, one-hot input: saliency = (Agg^T dz) W1, so its node average is (1/n_g)(sum_m w_m dz[m]) W1 -
                # one streaming reduction of dy with the BatchNorm-backward affine on load, then a [B, F] x [F, D] product
                if model.neighbor_pooling_type == "max":
                    # max pooling is not linear: the input gradient itself, then its average
                    _ops.bn_bwd_apply(u.z, u.mean, u.rstd, u.gamma, stats if use_batch else None, u.count, dy)
                    _ops.segment_weighted_colsum(max_pool_x_grad(dy, u.w, eps_l), bs.node_off, roi)
                    continue
                coef0 = bn_coef(u, stats, coef_ready)
                dz_sum = torch.empty(B, n_out, dtype=torch.float32, device=dev)
                _ops.segment_weighted_colsum(dy, bs.node_off, dz_sum, z=u.z if use_batch else None, coef=coef0,
                                             rowptr=bs.rowptr, mode=1 if average else 0, eps=eps_l)
                _ops.small_gemm(dz_sum, (dz_sum.stride(0), 1), u.w, (u.w.stride(0), 1), roi, B, n_in, n_out)
                continue
            if fused:
                # one pass: BatchNorm-backward apply (folded into the load as dz = A*dy + B*z + C), dW, db, dX and -
                # for an inner unit - the ReLU mask + BatchNorm-backward reduction of the unit below
                coef = bn_coef(u, stats, coef_ready, p2p)
                if j > 0:
                    p = units[j - 1]
                    dy_prev = torch.empty(M, n_in, dtype=torch.float32, device=dev)
                    stats_prev = zp.f64(2 * n_in)
                    coef_p, tail_p = _bn_backward_tail(p, stats_prev[0], comm)
                    took = _ops.linear_bwd(dy, u.z, coef, p.z, p.scale, p.shift, p.mean, p.rstd, u.w, dw, db, dy_prev,
                                           stats_prev[0], tail=tail_p)
                    ready = (dy_prev, stats_prev, coef_p if took is True else None)
                else:
                    dp = torch.empty(M, n_in, dtype=torch.float32, device=dev) if need_dp else None
                    _ops.linear_bwd(dy, u.z, coef, u.x_in, None, None, None, None, u.w, dw, db, dp, None)
                    if need_dp:
                        through_aggregation(layer, dp, eps_l)
                grads[gi], grads[gi + 1] = dw, db
                continue
            folded = False
            if gather0:
                g_agg = torch.empty(M, n_out, dtype=torch.float32, device=dev)
                if not learn_eps and not (need_x_grad and model.neighbor_pooling_type == "max"):
                    # layer-0 gather unit: dz is only ever aggregated, so the BatchNorm-backward apply rides on the
                    # aggregation kernel's row loads (dz = A*dy + B*z + C is never written); d bias follows in closed form
                    coef0 = bn_coef(u, stats, coef_ready)
                    folded = bool(bs.aggregate_affine(dy, u.z, coef0, g_agg, bwd_mode))
            if not folded:
                _ops.bn_bwd_apply(u.z, u.mean, u.rstd, u.gamma, stats if use_batch else None, u.count, dy)
            dz_u = dy                                                # now d loss / d z_j (unless folded)
            if j > 0:
                p = units[j - 1]
                _ops.linear_wgrad(dz_u, p.z, p.scale, p.shift, dw, db)
                dz = torch.empty(M, n_in, dtype=torch.float32, device=dev)
                _ops.linear(dz_u, u.w, True, None, None, None, dz, None)      # d a_{j-1} = dz_j @ W_j
                grads[gi], grads[gi + 1] = dw, db
                continue
            # ---- first unit of the layer: input is the neighbour aggregation --------------------
            if gather0:
                # z0 = Agg(W1^T[tags]) + b:  dW1^T[t] = sum_{tags[r]=t} (Agg^T dz)[r]
                if not folded:
                    bs.aggregate(dz_u, None, g_agg, bwd_mode, eps_l, None)
                dw1t = zp.f32(n_in, n_out)
                if bs.same_tags and n_out % 4 == 0:
                    _ops.rows_period_sum(g_agg, bs.uniform_n, bs.tags, dw1t)     # a streaming sum over the graphs
                else:
                    _ops.scatter_rows_add(g_agg, bs.tags, dw1t)
                dw = dw1t.t().contiguous()
                if folded:
                    # d bias = column sums of dz = A*sum(dy) + B*sum(z) + C*M. Under batch statistics that is identically
                    # zero (m1 = sum(dy)/M and sum(z) = M*mean cancel; the reference gets rounding noise); with running
                    # statistics B = C = 0 and it is A * sum(dy)
                    db = zp.f32(n_out) if use_batch else coef0[0] * stats[:n_out].to(torch.float32)
                else:
                    colsum, c_, o_ = zp.f64(2 * n_out)
                    _ops.col_stats(dz_u, colsum)                      # d bias = column sums of dz
                    from_f64.append((gi + 1, c_, o_, n_out, False))
                    db = None
                if learn_eps:
                    _ops.dot_rows(dz_u, sv.w1t, bs.tags, d_eps[layer:layer + 1])
                if need_x_grad and model.neighbor_pooling_type == "max":
                    d_x = max_pool_x_grad(dz_u, u.w, eps_l)
                elif need_x_grad:
                    d_x = torch.empty(M, n_in, dtype=torch.float32, device=dev)
                    _ops.linear(g_agg, u.w, True, None, None, None, d_x, None)   # (Agg^T dz) @ W1
            else:
                roi0 = layer == 0 and roi is not None
                if not roi0:
                    _ops.linear_wgrad(dz_u, u.x_in, None, None, dw, db)
                if need_dp:
                    dp = torch.empty(M, n_in, dtype=torch.float32, device=dev)
                    _ops.linear(dz_u, u.w, True, None, None, None, dp, None)
                    through_aggregation(layer, dp, eps_l)
            grads[gi], grads[gi + 1] = dw, db
    # float64 accumulators -> float32 gradients, one conversion per pool buffer (and one more for the shares of the
    # synchronised BatchNorm reductions: after the all-reduce those are sums over ALL ranks of gradients of each
    # rank's own mean loss; 1/world makes them this rank's share, so dist.average_gradients treats them like the rest)
    plain = [c.to(torch.float32) for c in zp.f64_chunks]
    if any(x[4] for x in from_f64):
        shared = [(c * (1.0 / comm.world)).to(torch.float32) for c in zp.f64_chunks]
    for gidx, c_, o_, n_, scaled in from_f64:
        g = (shared if scaled else plain)[c_][o_:o_ + n_]
        grads[gidx] = g.view(tuple(params[gidx].shape)) if gidx == 0 or gidx == 2 else g
    return d_x, grads


class GINFunction(torch.autograd.Function):
    """(g_f, d_logit) = GIN encoder + DGI scorer; see run_forward / run_backward."""

    @staticmethod
    def forward(ctx, runner, x_dense, *params):
        g_f, d_logit, sv = run_forward(runner.model, runner.bs, runner.neg_idx, runner.training, runner.with_dgi,
                                       x_dense.detach() if x_dense is not None else None,
                                       [p.detach() for p in params], runner.comm, max_padded=runner.max_padded)
        ctx.runner = runner
        ctx.sv = sv
        ctx.params = params
        ctx.need_x = x_dense is not None and x_dense.requires_grad
        if d_logit is None:
            d_logit = torch.zeros(0, 1, dtype=torch.float32, device=g_f.device)
        return g_f, d_logit

    @staticmethod
    def backward(ctx, dg_f, dd_logit):
        runner, sv = ctx.runner, ctx.sv
        if not sv.with_dgi:
            dd_logit = None
        need_x = ctx.need_x or runner.want_x_grad
        d_x, grads = run_backward(runner.model, sv, [p.detach() for p in ctx.params], dg_f, dd_logit, need_x,
                                  runner.comm, max_first=runner.max_first)
        runner.x_grad = d_x
        out = []
        for p, g in zip(ctx.params, grads):
            out.append(g if (g is not None and p.requires_grad) else None)
        return (None, d_x if ctx.need_x else None) + tuple(out)


class Runner(object):
    """Per-call context handed to GINFunction (non-tensor state)."""

    def __init__(self, model, bs, neg_idx, training, with_dgi, comm, want_x_grad=False):
        self.model = model
        self.bs = bs
        self.neg_idx = neg_idx
        self.training = training
        self.with_dgi = with_dgi
        self.comm = comm
        self.want_x_grad = want_x_grad
        self.max_first = None          # max pooling + input gradient: first neighbour-list entry per node (global ids)
        self.max_padded = None         # ... and the padded neighbour lists themselves ([M, W] int64, -1 pads)
        self.x_grad = None
