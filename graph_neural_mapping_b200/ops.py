"""Thin tensor-level wrappers over the C ABI (include/gnm.h).

Every function takes CUDA torch tensors (PyTorch is used for device memory and streams
only), extracts raw pointers / leading dimensions, enqueues the kernel on torch's current
stream and raises `RuntimeError` on a non-zero return code. There is no CPU path: a CPU
tensor is rejected.
"""
import ctypes

import torch

from . import lib as _libmod

_state = {"device": None}
LAUNCHES = [0]      # entry-point calls made through this module (an entry point may enqueue several kernels)
REPLAYED = [0]      # kernels launched by CUDA-graph replays (driver.Trainer / graphed.StepPlan account for them here)


def _lib():
    return _libmod.load()


def _stream(t):
    dev = t.device.index if t.device.index is not None else torch.cuda.current_device()
    if _state["device"] != dev:
        _libmod.check(_lib().gnm_set_device(dev), "gnm_set_device")
        _state["device"] = dev
    LAUNCHES[0] += 1
    return ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _ptr(t, dtype=None):
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("libgnm ops need CUDA tensors (there is no CPU fallback); got a %s tensor" % t.device)
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError("expected dtype %s, got %s" % (dtype, t.dtype))
    return ctypes.c_void_p(t.data_ptr())


def _mat(t):
    """(pointer, leading dimension) of a 2-D fp32 tensor whose rows are contiguous."""
    if t is None:
        return None, 0
    if t.dim() != 2 or (t.shape[1] > 1 and t.stride(1) != 1):
        raise RuntimeError("expected a row-major 2-D tensor, got shape %s strides %s" % (tuple(t.shape), t.stride()))
    return _ptr(t, torch.float32), int(t.stride(0))


def device_info():
    sm, ma, mi = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    smem = ctypes.c_int64()
    _libmod.check(_lib().gnm_device_info(ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi), ctypes.byref(smem)),
                  "gnm_device_info")
    return dict(sm_count=sm.value, cc=(ma.value, mi.value), smem_optin=smem.value)


KERNEL_FAMILIES = ("aggregate_csr", "aggregate_mma_sync", "aggregate_tc", "linear_ffma", "linear_tc", "linear_bwd_ffma",
                   "linear_bwd_dx_tc", "linear_wgrad_tc", "linear_wgrad_ffma", "other", "linear_bwd_onepass_tc",
                   "segment_colsum", "ig_expand", "ig_accumulate", "ig_attribute", "occlusion_expand")


def launch_counts():
    """Kernels libgnm has enqueued so far, per family (gnm_launch_counts of include/gnm.h) - which kernel family a
    code path really ran (tests) and how many kernels a step launches (bench.py). Host counters: a kernel recorded
    under CUDA-graph capture counts once."""
    buf = (ctypes.c_int64 * len(KERNEL_FAMILIES))()
    n = _lib().gnm_launch_counts(buf, len(KERNEL_FAMILIES))
    if n != len(KERNEL_FAMILIES):
        raise RuntimeError("gnm_launch_counts: library reports %d kernel families, binding expects %d" % (n, len(KERNEL_FAMILIES)))
    return {k: int(buf[i]) for i, k in enumerate(KERNEL_FAMILIES)}


def kernels_recorded():
    """Sum of libgnm's per-family launch counters: kernels ENQUEUED (or recorded under capture) so far."""
    return sum(launch_counts().values())


def kernels_launched():
    """libgnm kernels that have run (or are queued to run) on the device: eager launches plus CUDA-graph replays."""
    return kernels_recorded() + REPLAYED[0]


class _BnTailStruct(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int), ("count", ctypes.c_double), ("gamma", ctypes.c_void_p), ("beta", ctypes.c_void_p),
                ("eps", ctypes.c_float), ("momentum", ctypes.c_float), ("running_mean", ctypes.c_void_p),
                ("running_var", ctypes.c_void_p), ("num_batches_tracked", ctypes.c_void_p), ("scale", ctypes.c_void_p),
                ("shift", ctypes.c_void_p), ("mean", ctypes.c_void_p), ("rstd", ctypes.c_void_p), ("coef", ctypes.c_void_p),
                ("comm", ctypes.c_void_p), ("counter", ctypes.c_void_p)]


_TAIL_COUNTERS = {}


def _tail_counter(device):
    """One zero-initialised ticket per device: kernels of one stream run one after the other and leave it zero."""
    key = device.index if device.index is not None else torch.cuda.current_device()
    t = _TAIL_COUNTERS.get(key)
    if t is None:
        if torch.cuda.is_current_stream_capturing():
            # memory allocated under capture belongs to that graph's private pool and dies with it
            raise RuntimeError("the BatchNorm-tail ticket must exist before CUDA-graph capture (GraphStore creates it)")
        t = _TAIL_COUNTERS[key] = torch.zeros(1, dtype=torch.int32, device=device)
    return t


def prepare_device(device):
    """Per-device state that must exist before any CUDA-graph capture (called by engine.GraphStore)."""
    if device.type == "cuda":
        _tail_counter(device)


class BnTail(object):
    """gnm_bn_tail of include/gnm.h: the BatchNorm finalisation a stats-producing kernel runs in its last CTA."""

    FINALIZE, BWD_COEFFS = 1, 2

    def __init__(self, kind, count, gamma, mean, rstd, beta=None, eps=0.0, momentum=0.0, running_mean=None, running_var=None,
                 nbt=None, scale=None, shift=None, coef=None, p2p=None):
        dev = mean.device
        self.keep = (gamma, beta, running_mean, running_var, nbt, scale, shift, mean, rstd, coef, p2p, _tail_counter(dev))

        def a(t):
            return t.data_ptr() if t is not None else None
        self.struct = _BnTailStruct(int(kind), float(count), a(gamma), a(beta), float(eps), float(momentum), a(running_mean),
                                    a(running_var), a(nbt), a(scale), a(shift), a(mean), a(rstd), a(coef),
                                    ctypes.addressof(p2p.struct) if p2p is not None else None,
                                    _tail_counter(dev).data_ptr())

    def ref(self):
        return ctypes.byref(self.struct)


def _tail_ref(tail):
    return tail.ref() if tail is not None else None


# ---- structure ---------------------------------------------------------------------------

def csr_build(edges, edge_off, node_off, n_graphs, n_max, total_nodes, add_self_loops, local_cols):
    """edges int64 [2, E] (local ids), edge_off int64 [B+1], node_off int32 [B+1] -> rowptr, colidx, status."""
    e_total = int(edges.shape[1])
    edges = edges.contiguous()
    nnz = e_total + (total_nodes if add_self_loops else 0)
    if nnz >= 2 ** 31:
        raise RuntimeError("batch adjacency has %d entries; int32 CSR holds < 2^31" % nnz)
    dev = edges.device
    rowptr = torch.empty(total_nodes + 1, dtype=torch.int32, device=dev)
    colidx = torch.empty(max(nnz, 1), dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    _libmod.check(_lib().gnm_csr_build(_ptr(edges, torch.int64), e_total, _ptr(edge_off, torch.int64),
                                       _ptr(node_off, torch.int32), n_graphs, n_max, int(add_self_loops),
                                       int(local_cols), _ptr(rowptr), _ptr(colidx), _ptr(status), _stream(edges)),
                  "gnm_csr_build")
    return rowptr, colidx[:nnz], status


def csr_batch_gather(rp_addr, ci_addr, tag_addr, node_off, nnz_off, n_graphs, total_nodes, total_nnz, with_colidx=True):
    """with_colidx=False gathers row pointers (and tags) only and returns colidx = None."""
    dev = node_off.device
    rowptr = torch.empty(total_nodes + 1, dtype=torch.int32, device=dev)
    colidx = torch.empty(max(total_nnz, 1), dtype=torch.int32, device=dev) if with_colidx else None
    tags = torch.empty(total_nodes, dtype=torch.int32, device=dev) if tag_addr is not None else None
    _libmod.check(_lib().gnm_csr_batch_gather(_ptr(rp_addr, torch.int64), _ptr(ci_addr, torch.int64),
                                              _ptr(tag_addr, torch.int64) if tag_addr is not None else None,
                                              _ptr(node_off, torch.int32), _ptr(nnz_off, torch.int64), n_graphs,
                                              _ptr(rowptr), _ptr(colidx), _ptr(tags), _stream(node_off)),
                  "gnm_csr_batch_gather")
    return rowptr, (colidx[:total_nnz] if with_colidx else None), tags


# ---- aggregation -------------------------------------------------------------------------

def aggregate(rowptr, colidx, src, src_map, dst, mode, eps, bias=None):
    sp, lds = _mat(src)
    dp, ldd = _mat(dst)
    _libmod.check(_lib().gnm_aggregate(_ptr(rowptr, torch.int32), _ptr(colidx, torch.int32), int(dst.shape[0]),
                                       sp, lds, _ptr(src_map, torch.int32) if src_map is not None else None,
                                       dp, ldd, int(dst.shape[1]), int(mode), _ptr(eps, torch.float32),
                                       _ptr(bias, torch.float32), _stream(dst)), "gnm_aggregate")
    return dst


def bitmap_build(rowptr, colidx, node_off, bitmap_off, n_graphs, total_words):
    """Chunk CSR (local column ids) -> per-graph bitmaps (uint32 words as int32) + per-graph duplicate flags."""
    dev = rowptr.device
    bitmap = torch.empty(max(total_words, 1), dtype=torch.int32, device=dev)
    dup = torch.zeros(max(n_graphs, 1), dtype=torch.int32, device=dev)
    _libmod.check(_lib().gnm_bitmap_build(_ptr(rowptr, torch.int32), _ptr(colidx, torch.int32),
                                          _ptr(node_off, torch.int32), _ptr(bitmap_off, torch.int64), n_graphs,
                                          _ptr(bitmap), _ptr(dup), _stream(rowptr)), "gnm_bitmap_build")
    return bitmap, dup


DENSE_IMPL = [0]     # 0 auto, 1 mma.sync kernel, 2 tcgen05 kernel (A/B switch for tests and benchmarks)


def aggregate_tc_status():
    """True if a tcgen05 aggregation launch hit its bounded-wait timeout since the last call (device sync)."""
    v = ctypes.c_int(0)
    _libmod.check(_lib().gnm_aggregate_tc_status(ctypes.byref(v)), "gnm_aggregate_tc_status")
    return bool(v.value)


BN_ON_LOAD = True    # this module's aggregation and DGI entry points take bn_scale= / bn= (engine checks for it)


def aggregate_dense(bitmap_addr, node_off, rowptr, n_graphs, n_max, src, src_map, dst, mode, eps, bias=None, impl=None, *,
                    bn_scale=None, bn_shift=None, pooled=None, pool_scale=None):
    """dst = Agg(src) (include/gnm.h: gnm_aggregate_dense); returns dst. With bn_scale / bn_shift, src is the layer
    below's pre-BatchNorm output z and the kernel aggregates relu(z*bn_scale + bn_shift) without writing it, and pooled
    (optional, [B, >= F] view) receives that layer's graph readout (times pool_scale). Returns True then, or False with
    nothing launched when the batch does not fit that kernel (materialise h with bn_relu_readout instead)."""
    sp, lds = _mat(src)
    dp, ldd = _mat(dst)
    pp, ldp = _mat(pooled)
    on_load = bn_scale is not None
    rc = _lib().gnm_aggregate_dense(_ptr(bitmap_addr, torch.int64), _ptr(node_off, torch.int32),
                                    _ptr(rowptr, torch.int32), n_graphs, n_max, sp, lds,
                                    _ptr(src_map, torch.int32) if src_map is not None else None, dp, ldd,
                                    int(dst.shape[1]), int(mode), _ptr(eps, torch.float32),
                                    _ptr(bias, torch.float32), DENSE_IMPL[0] if impl is None else int(impl),
                                    _ptr(bn_scale, torch.float32), _ptr(bn_shift, torch.float32), pp, ldp,
                                    _ptr(pool_scale, torch.float32), _stream(dst))
    if on_load and rc in (-2, -3):          # GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN: not a tcgen05 batch
        LAUNCHES[0] -= 1
        return False
    _libmod.check(rc, "gnm_aggregate_dense")
    return True if on_load else dst


def aggregate_dense_table(bitmap_addr, node_off, rowptr, n_graphs, n_max, table, tags, dst, mode, eps, bias, out_stats,
                          tail=None):
    """z0 = Agg(table[tags]) (+ self term) + bias with one table shared by every graph, + column statistics of z0
    (include/gnm.h: gnm_aggregate_dense_table). Returns False, nothing launched, when the batch does not fit it."""
    tp, ldt = _mat(table)
    dp, ldd = _mat(dst)
    rc = _lib().gnm_aggregate_dense_table(_ptr(bitmap_addr, torch.int64), _ptr(node_off, torch.int32), _ptr(rowptr, torch.int32),
                                          n_graphs, n_max, tp, ldt, _ptr(tags, torch.int32), dp, ldd, int(dst.shape[1]),
                                          int(mode), _ptr(eps, torch.float32), _ptr(bias, torch.float32),
                                          _ptr(out_stats, torch.float64), _tail_ref(tail), _stream(dst))
    if rc in (-2, -3):
        LAUNCHES[0] -= 1
        return False
    _libmod.check(rc, "gnm_aggregate_dense_table")
    return True


TC_MAX_NODES = 416          # largest graph the tcgen05 aggregation kernel takes (gnm_aggregate_tc.cu)


def aggregate_dense_affine(bitmap_addr, node_off, rowptr, n_graphs, n_max, dy, z, coef, dst, mode):
    """dst = Agg(coef[0]*dy + coef[1]*z + coef[2]) on the tcgen05 kernel; returns False (nothing launched) when the
    batch does not fit that kernel - the caller then applies the affine with bn_bwd_apply and aggregates."""
    yp, ldy = _mat(dy)
    zp, ldz = _mat(z)
    dp, ldd = _mat(dst)
    rc = _lib().gnm_aggregate_dense_affine(_ptr(bitmap_addr, torch.int64), _ptr(node_off, torch.int32),
                                           _ptr(rowptr, torch.int32), n_graphs, n_max, yp, ldy, zp, ldz,
                                           _ptr(coef, torch.float32), dp, ldd, int(dst.shape[1]), int(mode), _stream(dst))
    if rc in (-2, -3):                      # GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN: not a tcgen05 batch
        LAUNCHES[0] -= 1
        return False
    _libmod.check(rc, "gnm_aggregate_dense_affine")
    return True


def aggregate_dense_relu_bn_bwd(bitmap_addr, node_off, rowptr, n_graphs, n_max, src, mode, eps, z, scale, shift, mean, rstd,
                                d_pooled, pool_scale, d_score, u, d_neg, n_neg, dy, stats, tail=None):
    """aggregate_dense(src) -> relu_bn_bwd_reduce(z, ...) in one tcgen05 kernel (the aggregated gradient is consumed in
    the copy-out). Returns False, with nothing launched, when the batch does not fit that kernel."""
    sp, lds = _mat(src)
    zp, ldz = _mat(z)
    gp, ldg = _mat(d_pooled)
    up, ldu = _mat(u)
    np_, ldn = _mat(d_neg)
    yp, ldy = _mat(dy)
    rc = _lib().gnm_aggregate_dense_relu_bn_bwd(_ptr(bitmap_addr, torch.int64), _ptr(node_off, torch.int32),
                                                _ptr(rowptr, torch.int32), n_graphs, n_max, sp, lds, int(dy.shape[1]),
                                                int(mode), _ptr(eps, torch.float32), zp, ldz, _ptr(scale), _ptr(shift),
                                                _ptr(mean), _ptr(rstd), gp, ldg, _ptr(pool_scale, torch.float32),
                                                _ptr(d_score, torch.float32), up, ldu, np_, ldn, int(n_neg), yp, ldy,
                                                _ptr(stats, torch.float64), _tail_ref(tail), _stream(dy))
    if rc in (-2, -3):                      # GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN: not a tcgen05 batch
        LAUNCHES[0] -= 1
        return False
    _libmod.check(rc, "gnm_aggregate_dense_relu_bn_bwd")
    return True


def dense_aggregate_ok(src, dst, bias=None):
    """Alignment contract of gnm_aggregate_dense (float4 row loads, float2 stores)."""
    return (dst.shape[1] % 4 == 0 and src.stride(0) % 4 == 0 and dst.stride(0) % 2 == 0 and
            src.data_ptr() % 16 == 0 and dst.data_ptr() % 16 == 0 and (bias is None or bias.data_ptr() % 16 == 0))


def dot_rows(a, b, b_map, out):
    ap, lda = _mat(a)
    bp, ldb = _mat(b)
    _libmod.check(_lib().gnm_dot_rows(ap, lda, bp, ldb, _ptr(b_map, torch.int32) if b_map is not None else None,
                                      int(a.shape[0]), int(a.shape[1]), _ptr(out, torch.float64), _stream(a)),
                  "gnm_dot_rows")
    return out


def scatter_rows_add(g, tags, table_grad):
    gp, ldg = _mat(g)
    tp, ldt = _mat(table_grad)
    need = int(_lib().gnm_scatter_rows_workspace(int(g.shape[0]), int(g.shape[1]), int(table_grad.shape[0])))
    ws = torch.empty(max(need, 1), dtype=torch.float32, device=g.device)
    _libmod.check(_lib().gnm_scatter_rows_add(gp, ldg, _ptr(tags, torch.int32), int(g.shape[0]), int(g.shape[1]),
                                              tp, ldt, int(table_grad.shape[0]), _ptr(ws), need, _stream(g)),
                  "gnm_scatter_rows_add")
    return table_grad


def rows_period_sum(g, period, tags, table_grad):
    """table_grad[tags[t]] += sum_k g[k*period + t] - scatter_rows_add for batches whose graphs all carry the same
    injective tag sequence (the caller checks that; tags = that sequence, or None for the identity)."""
    gp, ldg = _mat(g)
    tp, ldt = _mat(table_grad)
    need = int(_lib().gnm_rows_period_workspace(int(g.shape[0]), int(g.shape[1]), int(period)))
    ws = torch.empty(max(need, 1), dtype=torch.float32, device=g.device)
    _libmod.check(_lib().gnm_rows_period_sum(gp, ldg, int(g.shape[0]), int(g.shape[1]), int(period),
                                             _ptr(tags, torch.int32) if tags is not None else None, tp, ldt,
                                             int(table_grad.shape[0]), _ptr(ws), need, _stream(g)),
                  "gnm_rows_period_sum")
    return table_grad


def segment_weighted_colsum(x, node_off, out, z=None, coef=None, rowptr=None, mode=0, eps=None):
    """out[g] = (1/n_g) sum over graph g's rows m of w_m * v[m] (include/gnm.h: gnm_segment_weighted_colsum): v = x, or
    coef[0]*x + coef[1]*z + coef[2] with coef given (z None: coef[1] = coef[2] = 0); w_m = the row sums of the
    aggregation `mode` (0 sum, 1 average) with the optional eps self term as its backward applies them, or 1 without
    rowptr. out [B, W] may be a strided view. Returns out."""
    xp, ldx = _mat(x)
    zp, ldz = _mat(z)
    op, ldo = _mat(out)
    _libmod.check(_lib().gnm_segment_weighted_colsum(xp, ldx, zp, ldz, _ptr(coef, torch.float32), _ptr(node_off, torch.int32),
                                                     int(out.shape[0]), int(out.shape[1]), _ptr(rowptr, torch.int32),
                                                     int(mode), _ptr(eps, torch.float32), op, ldo, _stream(out)),
                  "gnm_segment_weighted_colsum")
    return out


# ---- integrated gradients: the virtual batch of path points (each real graph repeated `points` times, graph-major) ----

def ig_expand(p, bias, alpha, node_off, points, z):
    """z[(g, s, i)] = alpha[s] * p[node_off[g] + i] + bias (include/gnm.h: gnm_ig_expand): layer 0's output at every path
    point from one real-batch aggregation p. z is [points * p.shape[0], W]. Returns z."""
    pp, ldp = _mat(p)
    zp, ldz = _mat(z)
    _libmod.check(_lib().gnm_ig_expand(pp, ldp, _ptr(bias, torch.float32), _ptr(alpha, torch.float32),
                                       _ptr(node_off, torch.int32), int(node_off.shape[0]) - 1, int(p.shape[0]),
                                       int(points), int(p.shape[1]), zp, ldz, _stream(z)), "gnm_ig_expand")
    return z


def ig_accumulate(dy, coef, node_off, points, weight, out, accumulate):
    """out[r] (+)= weight * coef[0] o sum_s dy[(g, s, r - node_off[g])] (include/gnm.h: gnm_ig_accumulate): the
    quadrature sum of the path points' layer-0 gradients on the real rows, BatchNorm-backward (eval) on load. Returns out."""
    dp, ldd = _mat(dy)
    op, ldo = _mat(out)
    _libmod.check(_lib().gnm_ig_accumulate(dp, ldd, _ptr(coef, torch.float32), _ptr(node_off, torch.int32),
                                           int(node_off.shape[0]) - 1, int(out.shape[0]), int(points), int(out.shape[1]),
                                           float(weight), int(bool(accumulate)), op, ldo, _stream(out)),
                  "gnm_ig_accumulate")
    return out


def ig_attribute(t, table, tags, node_off, out):
    """out[g, d] = (1/n_g) sum over graph g's nodes n with tags[n] = d of <t[n], table[d]> (include/gnm.h:
    gnm_ig_attribute; NaN rows where t is not finite). out [B, D] may be a strided view. Returns out."""
    if table.shape[0] != out.shape[1]:
        raise RuntimeError("ig_attribute: table has %d rows, out %d columns" % (table.shape[0], out.shape[1]))
    tp, ldt = _mat(t)
    wp, ldw = _mat(table)
    op, ldo = _mat(out)
    _libmod.check(_lib().gnm_ig_attribute(tp, ldt, wp, ldw, int(out.shape[1]), _ptr(tags, torch.int32),
                                          _ptr(node_off, torch.int32), int(out.shape[0]), int(t.shape[1]), op, ldo,
                                          _stream(out)), "gnm_ig_attribute")
    return out


# ---- ROI occlusion: the virtual batch of occluded copies (each real graph repeated, graph-major) ----------------------

def occlusion_expand(p, bias, w1t, rowptr, colidx, tags, node_off, n_max, v_graph, v_tag, v_node_off, mode, eps, z):
    """z[v_node_off[v] + i] = p[m] + bias - c_d[m] * w1t[d], m = node_off[v_graph[v]] + i, d = v_tag[v] (include/gnm.h:
    gnm_occlusion_expand): layer 0's output for every occluded copy (v_tag >= 0) and baseline copy (v_tag < 0) of the
    real batch (rowptr, colidx with global ids, tags, node_off; n_max its largest graph) from one real-batch
    aggregation p. mode 0 sum, 1 average; eps [1] nullable (learn_eps). Returns z."""
    n_virtual = int(v_graph.shape[0])
    if v_tag.shape[0] != n_virtual or v_node_off.shape[0] != n_virtual + 1:
        raise RuntimeError("occlusion_expand: v_graph, v_tag and v_node_off describe %d, %d and %d virtual graphs"
                           % (n_virtual, v_tag.shape[0], v_node_off.shape[0] - 1))
    if w1t.shape[1] != p.shape[1] or z.shape[1] != p.shape[1]:
        raise RuntimeError("occlusion_expand: widths of p %d, w1t %d, z %d differ" % (p.shape[1], w1t.shape[1], z.shape[1]))
    pp, ldp = _mat(p)
    wp, ldw = _mat(w1t)
    zp, ldz = _mat(z)
    i32 = torch.int32
    _libmod.check(_lib().gnm_occlusion_expand(pp, ldp, _ptr(bias, torch.float32), wp, ldw, int(w1t.shape[0]),
                                              _ptr(rowptr, i32), _ptr(colidx, i32), _ptr(tags, i32), _ptr(node_off, i32),
                                              int(node_off.shape[0]) - 1, int(n_max), _ptr(v_graph, i32),
                                              _ptr(v_tag, i32), _ptr(v_node_off, i32), n_virtual, int(p.shape[1]),
                                              int(mode), _ptr(eps, torch.float32), zp, ldz, _stream(z)),
                  "gnm_occlusion_expand")
    return z


# ---- max pooling over neighbours ----------------------------------------------------------------

def col_min(h):
    """Packed (order-preserving key << 32 | first row) column minimum of h: the reference's dummy row (graphcnn.py:139-140)."""
    hp, ldh = _mat(h)
    packed = torch.full((int(h.shape[1]),), -1, dtype=torch.int64, device=h.device)       # all-ones
    _libmod.check(_lib().gnm_col_min(hp, ldh, int(h.shape[0]), int(h.shape[1]), _ptr(packed), _stream(h)), "gnm_col_min")
    return packed


def col_min_values(packed):
    """The float32 column minima held in the high words of col_min()'s packed keys (inverse of the order key)."""
    key = (packed >> 32) & 0xFFFFFFFF
    bits = torch.where((key & 0x80000000) != 0, key & 0x7FFFFFFF, (~key) & 0xFFFFFFFF)
    return _bits_to_float(bits)


def _bits_to_float(bits_i64):
    # int64 holding a 32-bit pattern -> float32 with that pattern
    lo = (bits_i64 & 0x7FFFFFFF).to(torch.int32)
    lo = torch.where((bits_i64 & 0x80000000) != 0, lo | torch.tensor(-0x80000000, dtype=torch.int32, device=bits_i64.device), lo)
    return lo.view(torch.float32)


def aggregate_max(rowptr, colidx, h, cmin, eps, out, argmax):
    hp, ldh = _mat(h)
    op, ldo = _mat(out)
    _libmod.check(_lib().gnm_aggregate_max(_ptr(rowptr, torch.int32), _ptr(colidx, torch.int32), int(h.shape[0]), hp, ldh,
                                           int(h.shape[1]), _ptr(cmin, torch.int64), _ptr(eps, torch.float32), op, ldo,
                                           _ptr(argmax, torch.int32), _stream(out)), "gnm_aggregate_max")
    return out


def aggregate_max_bwd(rowptr, colidx, d_out, argmax, cmin, eps, d_h):
    gp, ldg = _mat(d_out)
    dp, ldd = _mat(d_h)
    _libmod.check(_lib().gnm_aggregate_max_bwd(_ptr(rowptr, torch.int32), _ptr(colidx, torch.int32), int(d_out.shape[0]),
                                               gp, ldg, int(d_out.shape[1]), _ptr(argmax, torch.int32),
                                               _ptr(cmin, torch.int64), _ptr(eps, torch.float32), dp, ldd,
                                               _stream(d_h)), "gnm_aggregate_max_bwd")
    return d_h


# ---- peer-memory exchange (data parallel) ----------------------------------------------------

P2P_MAX_DOUBLES = 256
P2P_MAX_WORLD = 16


class _P2PStruct(ctypes.Structure):
    _fields_ = [("peers", ctypes.c_void_p), ("counter", ctypes.c_void_p), ("rank", ctypes.c_int), ("world", ctypes.c_int)]


class P2PComm(object):
    """gnm_p2p_comm of include/gnm.h: this rank's exchange buffer, its peers' buffers mapped through CUDA IPC, the
    device table of their addresses and the call counter. Built by dist.setup_p2p()."""

    def __init__(self, rank, world, device):
        self.rank, self.world, self.device = int(rank), int(world), device
        self.local = ctypes.c_void_p()
        handle = (ctypes.c_ubyte * 64)()
        _libmod.check(_lib().gnm_p2p_alloc(ctypes.byref(self.local), handle), "gnm_p2p_alloc")
        self.handle = bytes(handle)
        self.opened = []
        self.peers = None
        self.counter = torch.zeros(1, dtype=torch.int32, device=device)
        self.struct = None

    def connect(self, handles):
        addrs = []
        for r, h in enumerate(handles):
            if r == self.rank:
                addrs.append(self.local.value)
                continue
            ptr = ctypes.c_void_p()
            buf = (ctypes.c_ubyte * 64).from_buffer_copy(h)
            _libmod.check(_lib().gnm_p2p_open(buf, ctypes.byref(ptr)), "gnm_p2p_open")
            self.opened.append(ptr)
            addrs.append(ptr.value)
        self.peers = torch.tensor(addrs, dtype=torch.int64, device=self.device)
        self.struct = _P2PStruct(self.peers.data_ptr(), self.counter.data_ptr(), self.rank, self.world)

    def ref(self):
        return ctypes.byref(self.struct)

    def allreduce(self, t):
        """In-place sum over all ranks of a float64 tensor of at most P2P_MAX_DOUBLES elements."""
        _libmod.check(_lib().gnm_p2p_allreduce(_ptr(t, torch.float64), int(t.numel()), self.ref(), _stream(t)),
                      "gnm_p2p_allreduce")
        return t

    def status(self):
        v = ctypes.c_int(0)
        _libmod.check(_lib().gnm_p2p_status(ctypes.byref(v)), "gnm_p2p_status")
        return bool(v.value)

    def close(self):
        for ptr in self.opened:
            _lib().gnm_p2p_close(ptr, 0)
        self.opened = []
        if self.local is not None and self.local.value:
            _lib().gnm_p2p_close(self.local, 1)
            self.local = None


class _DevPtr(object):
    """A raw device pointer exposed through __cuda_array_interface__ so that torch can wrap it without copying."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(int(x) for x in shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}


class P2PRegion(object):
    """A peer-mapped memory region per rank (gnm_p2p_alloc_bytes + CUDA IPC): `tensor(r, ...)` is a torch view of rank
    r's region as mapped in THIS process - kernels read / write it through ordinary pointers over NVLink."""

    def __init__(self, rank, world, device, nbytes):
        self.rank, self.world, self.device, self.nbytes = int(rank), int(world), device, int(nbytes)
        self.local = ctypes.c_void_p()
        handle = (ctypes.c_ubyte * 64)()
        _libmod.check(_lib().gnm_p2p_alloc_bytes(ctypes.byref(self.local), handle, self.nbytes), "gnm_p2p_alloc_bytes")
        self.handle = bytes(handle)
        self.opened = []
        self.addrs = None
        self.bases = None            # device int64[world]: the regions' base addresses (gnm_p2p_push)
        self._views = {}

    def connect(self, handles):
        addrs = []
        for r, h in enumerate(handles):
            if r == self.rank:
                addrs.append(self.local.value)
                continue
            ptr = ctypes.c_void_p()
            buf = (ctypes.c_ubyte * 64).from_buffer_copy(h)
            _libmod.check(_lib().gnm_p2p_open(buf, ctypes.byref(ptr)), "gnm_p2p_open")
            self.opened.append(ptr)
            addrs.append(ptr.value)
        self.addrs = addrs
        self.bases = torch.tensor(addrs, dtype=torch.int64, device=self.device)

    def tensor(self, r, byte_offset, shape, dtype=torch.float32):
        key = (r, byte_offset, tuple(shape), dtype)
        t = self._views.get(key)
        if t is None:
            n = 1
            for d in shape:
                n *= int(d)
            esz = torch.empty(0, dtype=dtype).element_size()
            if byte_offset + n * esz > self.nbytes:
                raise RuntimeError("P2PRegion view of %d bytes at %d exceeds the region (%d)" % (n * esz, byte_offset, self.nbytes))
            typestr = {torch.float32: "<f4", torch.float64: "<f8", torch.int32: "<i4"}[dtype]
            t = torch.as_tensor(_DevPtr(self.addrs[r] + byte_offset, shape, typestr), device=self.device)
            self._views[key] = t
        return t

    def push(self, src, byte_offset):
        """src (float32, contiguous, numel % 4 == 0) -> every rank's region at byte_offset."""
        _libmod.check(_lib().gnm_p2p_push(_ptr(src, torch.float32), int(src.numel()), _ptr(self.bases, torch.int64), self.world,
                                          int(byte_offset), _stream(src)), "gnm_p2p_push")

    def close(self):
        self._views.clear()
        for ptr in self.opened:
            _lib().gnm_p2p_close(ptr, 0)
        self.opened = []
        if self.local is not None and self.local.value:
            _lib().gnm_p2p_close(self.local, 1)
            self.local = None


def sum_slots(base, world, stride, n, scale, out):
    _libmod.check(_lib().gnm_sum_slots(_ptr(base, torch.float32), int(world), int(stride), int(n), float(scale),
                                       _ptr(out, torch.float32), _stream(out)), "gnm_sum_slots")
    return out


def scatter_scaled_rows(idx, scale, src, dst):
    sp, lds = _mat(src)
    dp, ldd = _mat(dst)
    _libmod.check(_lib().gnm_scatter_scaled_rows(_ptr(idx, torch.int32), _ptr(scale, torch.float32), sp, lds, int(src.shape[0]),
                                                 int(src.shape[1]), dp, ldd, int(dst.shape[0]), _stream(src)),
                  "gnm_scatter_scaled_rows")
    return dst


# ---- MLP -----------------------------------------------------------------------------------

def set_linear_impl(impl):
    """0 auto, 1 fp32 FFMA kernel, 2 tcgen05 kernel (process-wide A/B switch)."""
    _libmod.check(_lib().gnm_set_linear_impl(int(impl)), "gnm_set_linear_impl")


def linear(x, w, w_is_kn, bias, in_scale, in_shift, y, col_stats, tail=None):
    """tail: BnTail(FINALIZE) run by the kernel's last CTA on col_stats. Returns True when the tail was taken; False
    when the shape runs on a kernel without tails (the Linear itself was still computed: call bn_finalize)."""
    xp, ldx = _mat(x)
    wp, ldw = _mat(w)
    yp, ldy = _mat(y)
    n_in = int(x.shape[1])
    n_out = int(y.shape[1])
    exp = (n_in, n_out) if w_is_kn else (n_out, n_in)
    if tuple(w.shape) != exp:
        raise RuntimeError("linear: weight shape %s does not match x %s -> y %s" % (tuple(w.shape), tuple(x.shape), tuple(y.shape)))
    args = (xp, ldx, int(x.shape[0]), n_in, wp, ldw, int(w_is_kn), _ptr(bias, torch.float32),
            _ptr(in_scale, torch.float32), _ptr(in_shift, torch.float32), yp, ldy, n_out, _ptr(col_stats, torch.float64))
    if tail is not None:
        rc = _lib().gnm_linear(*args, tail.ref(), _stream(y))
        if rc == 0:
            return True
        if rc != -2:
            _libmod.check(rc, "gnm_linear")
        LAUNCHES[0] -= 1                    # GNM_ERR_TOO_LARGE: nothing was launched, run without the tail
    _libmod.check(_lib().gnm_linear(*args, None, _stream(y)), "gnm_linear")
    return False


def linear_wgrad(dz, x, in_scale, in_shift, dw, dbias):
    zp, ldz = _mat(dz)
    xp, ldx = _mat(x)
    wp, ldw = _mat(dw)
    n_in = int(x.shape[1]) if x is not None else 0
    _libmod.check(_lib().gnm_linear_wgrad(zp, ldz, xp, ldx, int(dz.shape[0]), int(dz.shape[1]), n_in,
                                          _ptr(in_scale, torch.float32), _ptr(in_shift, torch.float32), wp, ldw,
                                          _ptr(dbias, torch.float32), _stream(dz)), "gnm_linear_wgrad")


def bn_bwd_coeffs(stats, count, gamma, mean, rstd, coef, p2p=None):
    """p2p: P2PComm - `stats` is all-reduced in place by the kernel before the coefficients are formed."""
    _libmod.check(_lib().gnm_bn_bwd_coeffs(_ptr(stats, torch.float64), float(count), _ptr(gamma, torch.float32),
                                           _ptr(mean), _ptr(rstd), _ptr(coef, torch.float32), int(mean.shape[0]),
                                           p2p.ref() if (p2p is not None and stats is not None) else None,
                                           _stream(coef)), "gnm_bn_bwd_coeffs")
    return coef


def linear_bwd(dy, z, coef, x, in_scale, in_shift, in_mean, in_rstd, w, dw, dbias, dx, stats_in, tail=None):
    """tail: BnTail(BWD_COEFFS) of the unit below, run on stats_in by the dx kernel's last CTA. Returns True when the tail
    was taken, False when the shape runs on the kernel without tails (the backward was still computed)."""
    yp, ldy = _mat(dy)
    zp, ldz = _mat(z)
    xp, ldx = _mat(x)
    wp, ldw = _mat(w)
    gp, ldg = _mat(dw)
    dp, ldd = _mat(dx)
    args = (yp, ldy, zp, ldz, _ptr(coef, torch.float32), xp, ldx, _ptr(in_scale), _ptr(in_shift), _ptr(in_mean), _ptr(in_rstd),
            wp, ldw, gp, ldg, _ptr(dbias, torch.float32), dp, ldd, _ptr(stats_in, torch.float64), int(dy.shape[0]),
            int(w.shape[0]), int(w.shape[1]))
    if tail is not None:
        rc = _lib().gnm_linear_bwd(*args, tail.ref(), _stream(dy))
        if rc == 0:
            return True
        if rc != -2:
            _libmod.check(rc, "gnm_linear_bwd")
        LAUNCHES[0] -= 1
    _libmod.check(_lib().gnm_linear_bwd(*args, None, _stream(dy)), "gnm_linear_bwd")
    return False


def col_stats(x, stats):
    xp, ldx = _mat(x)
    _libmod.check(_lib().gnm_col_stats(xp, ldx, int(x.shape[0]), int(x.shape[1]), _ptr(stats, torch.float64),
                                       _stream(x)), "gnm_col_stats")
    return stats


def bn_finalize(stats, count, gamma, beta, eps, momentum, running_mean, running_var, nbt, scale, shift, mean, rstd,
                p2p=None):
    """p2p: P2PComm whose ranks all call this in the same order - `stats` is then all-reduced in place by the kernel."""
    _libmod.check(_lib().gnm_bn_finalize(_ptr(stats, torch.float64), float(count), _ptr(gamma, torch.float32),
                                         _ptr(beta, torch.float32), float(eps), float(momentum),
                                         _ptr(running_mean, torch.float32), _ptr(running_var, torch.float32),
                                         _ptr(nbt, torch.int64), _ptr(scale), _ptr(shift), _ptr(mean), _ptr(rstd),
                                         int(scale.shape[0]), p2p.ref() if p2p is not None else None,
                                         _stream(scale)), "gnm_bn_finalize")


def bn_eval_affine(running_mean, running_var, gamma, beta, eps, scale, shift, mean, rstd):
    _libmod.check(_lib().gnm_bn_eval_affine(_ptr(running_mean, torch.float32), _ptr(running_var, torch.float32),
                                            _ptr(gamma, torch.float32), _ptr(beta, torch.float32), float(eps),
                                            _ptr(scale), _ptr(shift), _ptr(mean), _ptr(rstd), int(scale.shape[0]),
                                            _stream(scale)), "gnm_bn_eval_affine")


def bn_relu_readout(z, scale, shift, h, node_off, n_graphs, pool_scale, pooled):
    zp, ldz = _mat(z)
    hp, ldh = _mat(h)
    pp, ldp = _mat(pooled)
    _libmod.check(_lib().gnm_bn_relu_readout(zp, ldz, int(z.shape[0]), int(z.shape[1]), _ptr(scale), _ptr(shift),
                                             hp, ldh, _ptr(node_off, torch.int32), n_graphs,
                                             _ptr(pool_scale, torch.float32), pp, ldp, _stream(z)),
                  "gnm_bn_relu_readout")


def relu_bn_bwd_reduce(z, scale, shift, mean, rstd, d_out, d_pooled, pool_scale, d_score, u, d_neg, n_neg,
                       node_off, n_graphs, dy, stats, tail=None):
    """Returns True when `tail` (BnTail BWD_COEFFS) was run by the kernel's last CTA."""
    zp, ldz = _mat(z)
    op, ldo = _mat(d_out)
    gp, ldg = _mat(d_pooled)
    up, ldu = _mat(u)
    np_, ldn = _mat(d_neg)
    yp, ldy = _mat(dy)
    args = (zp, ldz, int(z.shape[0]), int(z.shape[1]), _ptr(scale), _ptr(shift), _ptr(mean), _ptr(rstd), op, ldo, gp, ldg,
            _ptr(pool_scale, torch.float32), _ptr(d_score, torch.float32), up, ldu, np_, ldn, int(n_neg),
            _ptr(node_off, torch.int32), n_graphs, yp, ldy, _ptr(stats, torch.float64))
    if tail is not None:
        rc = _lib().gnm_relu_bn_bwd_reduce(*args, tail.ref(), _stream(z))
        if rc == 0:
            return True
        if rc != -2:
            _libmod.check(rc, "gnm_relu_bn_bwd_reduce")
        LAUNCHES[0] -= 1
    _libmod.check(_lib().gnm_relu_bn_bwd_reduce(*args, None, _stream(z)), "gnm_relu_bn_bwd_reduce")
    return False


def bn_bwd_apply(z, mean, rstd, gamma, stats, count, dy):
    zp, ldz = _mat(z)
    yp, ldy = _mat(dy)
    _libmod.check(_lib().gnm_bn_bwd_apply(zp, ldz, int(dy.shape[0]), int(dy.shape[1]), _ptr(mean), _ptr(rstd),
                                          _ptr(gamma, torch.float32), _ptr(stats, torch.float64), float(count), yp, ldy,
                                          _stream(dy)), "gnm_bn_bwd_apply")


# ---- DGI -----------------------------------------------------------------------------------

def _hall(h_all):
    if h_all.dim() != 3 or h_all.stride(2) != 1:
        raise RuntimeError("h_all must be [L, M, F] with contiguous rows")
    return _ptr(h_all, torch.float32), int(h_all.stride(0)), int(h_all.shape[0]), int(h_all.shape[2]), int(h_all.stride(1))


def _bn_table(bn, h_all):
    """bn: None, or per-layer scale | shift as an [L, >= 2, F] view with contiguous rows (e.g. the first two rows of each
    layer's [4, F] BatchNorm buffers): h_all then holds the pre-BatchNorm z and h = relu(z*scale + shift) on load."""
    if bn is None:
        return None, 0
    if (bn.dim() != 3 or bn.shape[0] != h_all.shape[0] or bn.shape[1] < 2 or bn.shape[2] != h_all.shape[2] or
            bn.stride(2) != 1 or bn.stride(1) != bn.shape[2] or bn.dtype != torch.float32):
        raise RuntimeError("bn must be an [L, 2, F] float32 table with contiguous scale | shift rows")
    return _ptr(bn), int(bn.stride(0))


def gather_nf_rows(h_all, n_rows, out=None, bn=None):
    hp, ls, nl, nf, ldh = _hall(h_all)
    bp, ldb = _bn_table(bn, h_all)
    table = out if out is not None else torch.empty(n_rows, nl * nf, dtype=torch.float32, device=h_all.device)
    if tuple(table.shape) != (n_rows, nl * nf) or not table.is_contiguous():
        raise RuntimeError("gather_nf_rows: out must be a contiguous [%d, %d] tensor" % (n_rows, nl * nf))
    _libmod.check(_lib().gnm_gather_nf_rows(hp, ls, nl, nf, ldh, n_rows, bp, ldb, _ptr(table), _stream(h_all)),
                  "gnm_gather_nf_rows")
    return table


def dgi_score_fwd(h_all, u, neg_table, neg_idx, node_off, n_graphs, bias, out, bn=None):
    hp, ls, nl, nf, ldh = _hall(h_all)
    bp, ldb = _bn_table(bn, h_all)
    _libmod.check(_lib().gnm_dgi_score_fwd(hp, ls, nl, nf, ldh, int(h_all.shape[1]), _ptr(u.contiguous(), torch.float32),
                                           _ptr(neg_table, torch.float32), _ptr(neg_idx, torch.int32),
                                           _ptr(node_off, torch.int32), n_graphs, _ptr(bias, torch.float32), bp, ldb,
                                           _ptr(out, torch.float32), _stream(out)), "gnm_dgi_score_fwd")
    return out


def dgi_score_bwd(h_all, d_out, neg_table, neg_idx, node_off, n_graphs, du, s2, d_bias, bn=None):
    hp, ls, nl, nf, ldh = _hall(h_all)
    bp, ldb = _bn_table(bn, h_all)
    _libmod.check(_lib().gnm_dgi_score_bwd(hp, ls, nl, nf, ldh, int(h_all.shape[1]), _ptr(d_out, torch.float32),
                                           _ptr(neg_table, torch.float32), _ptr(neg_idx, torch.int32),
                                           _ptr(node_off, torch.int32), n_graphs, bp, ldb, _ptr(du, torch.float32),
                                           _ptr(s2, torch.float32), _ptr(d_bias, torch.float64), _stream(du)),
                  "gnm_dgi_score_bwd")


def dgi_score_train(h_all, u, neg_table, neg_idx, node_off, n_graphs, bias, grad_scale, loss_scale, out, d_score, du, s2,
                    d_bias, loss_acc, bn=None):
    """dgi_score_fwd + bce_logits + dgi_score_bwd in one pass (include/gnm.h: gnm_dgi_score_train). Returns False, with
    nothing launched, when the shape does not fit the kernel - make the three calls then."""
    hp, ls, nl, nf, ldh = _hall(h_all)
    bp, ldb = _bn_table(bn, h_all)
    rc = _lib().gnm_dgi_score_train(hp, ls, nl, nf, ldh, int(h_all.shape[1]), _ptr(u.contiguous(), torch.float32),
                                    _ptr(neg_table, torch.float32), _ptr(neg_idx, torch.int32), _ptr(node_off, torch.int32),
                                    n_graphs, _ptr(bias, torch.float32), bp, ldb, float(grad_scale), float(loss_scale),
                                    _ptr(out, torch.float32), _ptr(d_score, torch.float32), _ptr(du, torch.float32),
                                    _ptr(s2, torch.float32), _ptr(d_bias, torch.float64), _ptr(loss_acc, torch.float64),
                                    _stream(out))
    if rc in (-2, -3):                      # GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN: not the kernel's shape
        LAUNCHES[0] -= 1
        return False
    _libmod.check(rc, "gnm_dgi_score_train")
    return True


def rowdot_score(h, u, rows_per_graph, bias, s_bias, out):
    hp, ldh = _mat(h)
    up, ldu = _mat(u)
    _libmod.check(_lib().gnm_rowdot_score(hp, ldh, int(h.shape[0]), int(h.shape[1]), up, ldu, int(rows_per_graph),
                                          _ptr(bias, torch.float32), _ptr(s_bias, torch.float32),
                                          _ptr(out, torch.float32), _stream(out)), "gnm_rowdot_score")
    return out


# ---- the [B, L*F]-sized remainder of a training step (gnm_train.cu) ---------------------------

def _ptr_array(tensors, dtype=torch.float32):
    arr = (ctypes.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        if not t.is_cuda or t.dtype != dtype or not t.is_contiguous():
            raise RuntimeError("expected contiguous CUDA %s tensors" % dtype)
        arr[i] = t.data_ptr()
    return arr


def heads_ce(g_f, weights, biases, mask, labels, inv_count, c_logit, loss_acc, d_gf, d_weights, d_biases, workspace, counter):
    """graphcnn.py:228-231 + nn.CrossEntropyLoss forward and backward (see include/gnm.h: gnm_heads_ce)."""
    gp, ldg = _mat(g_f)
    dp, ldd = _mat(d_gf)
    n_layers, n_classes, n_feat = len(weights), int(weights[0].shape[0]), int(weights[0].shape[1])
    _libmod.check(_lib().gnm_heads_ce(gp, ldg, int(g_f.shape[0]), n_layers, n_feat, n_classes, _ptr_array(weights),
                                      _ptr_array(biases), _ptr(mask, torch.float32), _ptr(labels, torch.int64),
                                      float(inv_count), _ptr(c_logit, torch.float32), _ptr(loss_acc, torch.float64), dp, ldd,
                                      _ptr_array(d_weights), _ptr_array(d_biases), _ptr(workspace, torch.float32),
                                      int(workspace.numel()), _ptr(counter, torch.int32), _stream(g_f)), "gnm_heads_ce")


def heads_fwd(g_f, weights, biases, mask, c_logit):
    gp, ldg = _mat(g_f)
    n_layers, n_classes, n_feat = len(weights), int(weights[0].shape[0]), int(weights[0].shape[1])
    _libmod.check(_lib().gnm_heads_fwd(gp, ldg, int(g_f.shape[0]), n_layers, n_feat, n_classes, _ptr_array(weights),
                                       _ptr_array(biases), _ptr(mask, torch.float32), _ptr(c_logit, torch.float32),
                                       _stream(g_f)), "gnm_heads_fwd")
    return c_logit


def heads_bwd(g_f, weights, mask, d_logit, d_gf, d_weights, d_biases, workspace, counter):
    gp, ldg = _mat(g_f)
    dp, ldd = _mat(d_gf)
    n_layers, n_classes, n_feat = len(weights), int(weights[0].shape[0]), int(weights[0].shape[1])
    _libmod.check(_lib().gnm_heads_bwd(gp, ldg, int(g_f.shape[0]), n_layers, n_feat, n_classes, _ptr_array(weights),
                                       _ptr(mask, torch.float32), _ptr(d_logit, torch.float32), dp, ldd, _ptr_array(d_weights),
                                       _ptr_array(d_biases), _ptr(workspace, torch.float32), int(workspace.numel()),
                                       _ptr(counter, torch.int32), _stream(g_f)), "gnm_heads_bwd")


def heads_ce_workspace(n_graphs, n_layers, n_feat, n_classes):
    return int(_lib().gnm_heads_ce_workspace(int(n_graphs), int(n_layers), int(n_feat), int(n_classes)))


def bce_logits(logits, n_pos, grad_scale, loss_scale, loss_acc, d_logits):
    _libmod.check(_lib().gnm_bce_logits(_ptr(logits, torch.float32), int(logits.numel()), int(n_pos), float(grad_scale),
                                        float(loss_scale), _ptr(loss_acc, torch.float64), _ptr(d_logits, torch.float32),
                                        _stream(logits)), "gnm_bce_logits")


def small_gemm(a, a_strides, b, b_strides, c, m, n, k, sigmoid_a_out=None, dsig_s=None, dsig_add=None):
    """C[m,n] = sum_k A(m,k) B(k,n) with element strides (sam, sak) / (sbk, sbn); see include/gnm.h: gnm_small_gemm."""
    cp, ldc = _mat(c)
    ao, ldao = _mat(sigmoid_a_out)
    sp, lds = _mat(dsig_s)
    dp, ldadd = _mat(dsig_add)
    _libmod.check(_lib().gnm_small_gemm(_ptr(a, torch.float32), int(a_strides[0]), int(a_strides[1]), _ptr(b, torch.float32),
                                        int(b_strides[0]), int(b_strides[1]), cp, ldc, int(m), int(n), int(k),
                                        1 if sigmoid_a_out is not None else 0, ao, ldao, sp, lds, dp, ldadd, _stream(c)),
                  "gnm_small_gemm")
    return c


def dgi_neg_grad(neg_idx, s2, u, d_neg):
    up, ldu = _mat(u)
    dp, ldn = _mat(d_neg)
    _libmod.check(_lib().gnm_dgi_neg_grad(_ptr(neg_idx, torch.int32), _ptr(s2, torch.float32), up, ldu, int(u.shape[0]),
                                          int(u.shape[1]), dp, ldn, int(d_neg.shape[0]), _stream(d_neg)), "gnm_dgi_neg_grad")
    return d_neg


def adam_step(params, grads, state_off, exp_avg, exp_avg_sq, step, lr, beta1, beta2, eps, weight_decay, grad_scale,
              loss_terms=None, loss_out=None):
    """torch.optim.Adam over a table of tensors in one launch (include/gnm.h: gnm_adam_step)."""
    n = len(params)
    numel = (ctypes.c_int32 * n)(*[int(p.numel()) for p in params])
    offs = (ctypes.c_int32 * n)(*[int(o) for o in state_off])
    _libmod.check(_lib().gnm_adam_step(_ptr_array(params), _ptr_array(grads), numel, offs, n, _ptr(exp_avg, torch.float32),
                                       _ptr(exp_avg_sq, torch.float32), _ptr(step, torch.float32), _ptr(lr, torch.float32),
                                       float(beta1), float(beta2), float(eps), float(weight_decay), float(grad_scale),
                                       _ptr(loss_terms, torch.float64), int(loss_terms.numel()) if loss_terms is not None else 0,
                                       _ptr(loss_out, torch.float32), _stream(exp_avg)), "gnm_adam_step")
