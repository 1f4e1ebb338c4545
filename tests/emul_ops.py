"""A CPU stand-in for `graph_neural_mapping_b200.ops`, for HOST-LOGIC tests only.

It lives under tests/ and is injected with monkeypatch; the product path cannot reach it.
Each function follows the contract written in include/gnm.h (not the kernels' code), using
plain torch CPU ops, so that the orchestration in `engine.py` (the hand-derived backward, the
graph store, the data-parallel exchanges) can be checked against the golden fixtures without
a GPU. The CUDA kernels themselves are checked by the `-m gpu` tests.
"""
import ctypes

import numpy as np
import torch


def _i32_at(addr, n):
    if n == 0:
        return np.zeros(0, dtype=np.int32)
    return np.ctypeslib.as_array(ctypes.cast(int(addr), ctypes.POINTER(ctypes.c_int32)), shape=(n,))


def device_info():
    return dict(sm_count=0, cc=(0, 0), smem_optin=0)


def csr_build(edges, edge_off, node_off, n_graphs, n_max, total_nodes, add_self_loops, local_cols):
    e = edges.numpy().reshape(2, -1)
    eo, no = edge_off.numpy(), node_off.numpy().astype(np.int64)
    rows, cols, bad = [], [], 0
    for g in range(n_graphs):
        s, d = e[0, eo[g]:eo[g + 1]], e[1, eo[g]:eo[g + 1]]
        n = no[g + 1] - no[g]
        ok = (s >= 0) & (s < n) & (d >= 0) & (d < n)
        bad |= int((~ok).any())
        s, d = s[ok], d[ok]
        if add_self_loops:
            s = np.concatenate([s, np.arange(n)])
            d = np.concatenate([d, np.arange(n)])
        order = np.lexsort((d, s))
        rows.append(s[order] + no[g])
        cols.append(d[order] + (0 if local_cols else no[g]))
    rows = np.concatenate(rows) if rows else np.zeros(0, dtype=np.int64)
    cols = np.concatenate(cols) if cols else np.zeros(0, dtype=np.int64)
    rowptr = np.zeros(total_nodes + 1, dtype=np.int64)
    np.add.at(rowptr, rows + 1, 1)
    rowptr = np.cumsum(rowptr)
    return (torch.from_numpy(rowptr.astype(np.int32)), torch.from_numpy(cols.astype(np.int32)),
            torch.tensor([bad], dtype=torch.int32))


def csr_batch_gather(rp_addr, ci_addr, tag_addr, node_off, nnz_off, n_graphs, total_nodes, total_nnz, with_colidx=True):
    no, zo = node_off.numpy(), nnz_off.numpy()
    rowptr = np.zeros(total_nodes + 1, dtype=np.int32)
    colidx = np.zeros(total_nnz, dtype=np.int32)
    tags = np.zeros(total_nodes, dtype=np.int32) if tag_addr is not None else None
    for g in range(n_graphs):
        n = int(no[g + 1] - no[g])
        rp = _i32_at(rp_addr[g], n + 1)
        nnz = int(rp[n] - rp[0])
        ci = _i32_at(ci_addr[g], nnz)
        rowptr[no[g]:no[g] + n] = rp[:n] - rp[0] + zo[g]
        colidx[zo[g]:zo[g] + nnz] = ci + no[g]
        if tags is not None:
            tags[no[g]:no[g] + n] = _i32_at(tag_addr[g], n)
    rowptr[total_nodes] = total_nnz
    return (torch.from_numpy(rowptr), torch.from_numpy(colidx) if with_colidx else None,
            torch.from_numpy(tags) if tags is not None else None)


def _csr(rowptr, colidx, m):
    return torch.sparse_csr_tensor(rowptr.long(), colidx.long(), torch.ones(colidx.numel(), dtype=torch.float64),
                                   size=(m, m)).to_dense()


def aggregate(rowptr, colidx, src, src_map, dst, mode, eps, bias=None):
    m = dst.shape[0]
    a = _csr(rowptr, colidx, m)
    s = src.double()
    if src_map is not None:
        s = s[src_map.long()]
    deg = a.sum(1, keepdim=True)
    if mode == 2:
        # an isolated node (deg 0) is never gathered, so its scale is irrelevant
        out = a @ (s / deg.clamp(min=1))
    else:
        out = a @ s
        if mode == 1:
            out = out / deg
    if eps is not None:
        out = out + (1 + eps.double()) * s
    if bias is not None:
        out = out + bias.double()
    dst.copy_(out.float())
    return dst


def bitmap_build(rowptr, colidx, node_off, bitmap_off, n_graphs, total_words):
    rp, ci, no, bo = rowptr.numpy(), colidx.numpy(), node_off.numpy(), bitmap_off.numpy()
    bm = np.zeros(max(total_words, 1), dtype=np.uint32)
    dup = np.zeros(max(n_graphs, 1), dtype=np.int32)
    for g in range(n_graphs):
        n = int(no[g + 1] - no[g])
        w = (n + 31) // 32
        for r in range(n):
            cols = ci[rp[no[g] + r]:rp[no[g] + r + 1]]
            if len(np.unique(cols)) != len(cols):
                dup[g] = 1
            for c in cols:
                bm[bo[g] + r * w + (c >> 5)] |= np.uint32(1) << np.uint32(c & 31)
    return torch.from_numpy(bm.view(np.int32)), torch.from_numpy(dup)


def dense_aggregate_ok(src, dst, bias=None):
    return dst.shape[1] % 4 == 0


def aggregate_dense_relu_bn_bwd(bitmap_addr, node_off, rowptr, n_graphs, n_max, src, mode, eps, z, scale, shift, mean, rstd,
                                d_pooled, pool_scale, d_score, u, d_neg, n_neg, dy, stats, tail=None):
    if n_max > 416 or dy.shape[1] > 64:
        return False
    d_h = torch.empty_like(dy)
    aggregate_dense(bitmap_addr, node_off, rowptr, n_graphs, n_max, src, None, d_h, mode, eps)
    relu_bn_bwd_reduce(z, scale, shift, mean, rstd, d_h, d_pooled, pool_scale, d_score, u, d_neg, n_neg, node_off, n_graphs,
                       dy, stats)
    return True


def aggregate_dense_affine(bitmap_addr, node_off, rowptr, n_graphs, n_max, dy, z, coef, dst, mode):
    if n_max > 416:
        return False
    dz = (coef[0].double() * dy.double() + coef[1].double() * z.double() + coef[2].double()).to(dy.dtype)
    aggregate_dense(bitmap_addr, node_off, rowptr, n_graphs, n_max, dz, None, dst, mode, None)
    return True


def aggregate_dense(bitmap_addr, node_off, rowptr, n_graphs, n_max, src, src_map, dst, mode, eps, bias=None, impl=None):
    """Contract of gnm_aggregate_dense: the adjacency is read from the per-graph bitmaps."""
    no = node_off.numpy()
    m = dst.shape[0]
    a = torch.zeros(m, m, dtype=torch.float64)
    for g in range(n_graphs):
        n = int(no[g + 1] - no[g])
        w = (n + 31) // 32
        words = _i32_at(bitmap_addr[g], n * w).view(np.uint32).reshape(n, w)
        bits = ((words[:, :, None] >> np.arange(32, dtype=np.uint32)[None, None, :]) & 1).reshape(n, w * 32)[:, :n]
        a[no[g]:no[g] + n, no[g]:no[g] + n] = torch.from_numpy(bits.astype(np.float64))
    s = src.double()
    if src_map is not None:
        s = s[src_map.long()]
    deg = a.sum(1, keepdim=True)
    if mode == 2:
        out = a @ (s / deg.clamp(min=1))
    else:
        out = a @ s
        if mode == 1:
            out = out / deg
    if eps is not None:
        out = out + (1 + eps.double()) * s
    if bias is not None:
        out = out + bias.double()
    dst.copy_(out.float())
    return dst


def dot_rows(a, b, b_map, out):
    bb = b if b_map is None else b[b_map.long()]
    out += (a.double() * bb.double()).sum()
    return out


def scatter_rows_add(g, tags, table_grad):
    table_grad.index_add_(0, tags.long(), g)
    return table_grad


def col_min(h):
    """Stand-in keeps (values, first argmin rows) as a tuple instead of the packed device words."""
    v, _ = h.min(0)
    first = (h == v.unsqueeze(0)).float().argmax(0)
    return (v, first)


def col_min_values(cmin):
    return cmin[0]


def aggregate_max(rowptr, colidx, h, cmin, eps, out, argmax):
    m, f = h.shape
    rp, ci = rowptr.long(), colidx.long()
    for i in range(m):
        nb = ci[rp[i]:rp[i + 1]]
        if nb.numel() == 0:
            out[i] = cmin[0]
            argmax[i] = m
        else:
            vals = h[nb]                                            # [deg, f], ascending column order
            best = vals.max(0).values
            first = (vals == best.unsqueeze(0)).float().argmax(0)   # lowest column id among ties
            out[i] = best
            argmax[i] = nb[first].to(argmax.dtype)
        if eps is not None:
            out[i] += (1.0 + eps[0]) * h[i]
    return out


def aggregate_max_bwd(rowptr, colidx, d_out, argmax, cmin, eps, d_h):
    m, f = d_out.shape
    d_h.zero_()
    cols = torch.arange(f)
    for i in range(m):
        src = argmax[i].long()
        real = src < m
        d_h[src[real], cols[real]] += d_out[i, real]
        if (~real).any():
            d_h[cmin[1][~real], cols[~real]] += d_out[i, ~real]
    if eps is not None:
        d_h += (1.0 + eps[0]) * d_out
    return d_h


def rows_period_sum(g, period, tags, table_grad):
    s = g.view(-1, period, g.shape[1]).double().sum(0).to(g.dtype)
    idx = torch.arange(period) if tags is None else tags[:period].long()
    ok = (idx >= 0) & (idx < table_grad.shape[0])
    table_grad.index_add_(0, idx[ok], s[ok])
    return table_grad


def _act(x, sc, sh):
    return x if sc is None else torch.relu(x * sc + sh)


def linear(x, w, w_is_kn, bias, in_scale, in_shift, y, col_stats, tail=None):
    a = _act(x, in_scale, in_shift).double()
    out = a @ (w.double() if w_is_kn else w.double().t())
    if bias is not None:
        out = out + bias.double()
    y.copy_(out.float())
    if col_stats is not None:
        n = y.shape[1]
        col_stats[:n] += y.double().sum(0)
        col_stats[n:] += (y.double() ** 2).sum(0)
    return False            # no BatchNorm tail taken (ops.linear's contract)


def linear_wgrad(dz, x, in_scale, in_shift, dw, dbias):
    if x is not None:
        dw += (dz.double().t() @ _act(x, in_scale, in_shift).double()).float()
    if dbias is not None:
        dbias += dz.double().sum(0).float()


def bn_bwd_coeffs(stats, count, gamma, mean, rstd, coef, p2p=None):
    f = mean.shape[0]
    g = gamma * rstd
    coef[0] = g
    if stats is None:
        coef[1] = 0
        coef[2] = 0
    else:
        m1, m2 = (stats[:f] / count).float(), (stats[f:] / count).float()
        coef[1] = -g * rstd * m2
        coef[2] = g * (rstd * m2 * mean - m1)
    return coef


def linear_bwd(dy, z, coef, x, in_scale, in_shift, in_mean, in_rstd, w, dw, dbias, dx, stats_in, tail=None):
    dz = (coef[0] * dy + coef[1] * z + coef[2]).double()
    a = _act(x, in_scale, in_shift).double()
    dw += (dz.t() @ a).float()
    if dbias is not None:
        dbias += dz.sum(0).float()
    if dx is not None or stats_in is not None:
        g = dz @ w.double()
        if in_scale is not None:
            g = torch.where(a > 0, g, torch.zeros_like(g))
        if dx is not None:
            dx.copy_(g.float())
        if stats_in is not None:
            n = x.shape[1]
            stats_in[:n] += g.sum(0)
            stats_in[n:] += (g * ((x - in_mean) * in_rstd).double()).sum(0)


def col_stats(x, stats):
    n = x.shape[1]
    stats[:n] += x.double().sum(0)
    stats[n:] += (x.double() ** 2).sum(0)
    return stats


def bn_finalize(stats, count, gamma, beta, eps, momentum, running_mean, running_var, nbt, scale, shift, mean, rstd,
                p2p=None):
    n = scale.shape[0]
    mu = stats[:n] / count
    var = (stats[n:] / count - mu * mu).clamp_(min=0)
    r = 1.0 / torch.sqrt(var + eps)
    scale.copy_((gamma.double() * r).float())
    shift.copy_(beta - mu.float() * scale)
    mean.copy_(mu.float())
    rstd.copy_(r.float())
    if running_mean is not None:
        running_mean.mul_(1 - momentum).add_(momentum * mu.float())
    if running_var is not None:
        unb = var * (count / (count - 1)) if count > 1 else var
        running_var.mul_(1 - momentum).add_(momentum * unb.float())
    if nbt is not None:
        nbt += 1


def bn_eval_affine(running_mean, running_var, gamma, beta, eps, scale, shift, mean, rstd):
    r = 1.0 / torch.sqrt(running_var + eps)
    scale.copy_(gamma * r)
    shift.copy_(beta - running_mean * scale)
    mean.copy_(running_mean)
    rstd.copy_(r)


def _graph_of_row(node_off, m):
    no = node_off.long()
    return torch.repeat_interleave(torch.arange(no.numel() - 1), no[1:] - no[:-1])


def bn_relu_readout(z, scale, shift, h, node_off, n_graphs, pool_scale, pooled):
    v = torch.relu(z * scale + shift)
    if h is not None:
        h.copy_(v)
    if pooled is not None:
        gid = _graph_of_row(node_off, z.shape[0])
        out = torch.zeros(n_graphs, z.shape[1], dtype=torch.float64).index_add_(0, gid, v.double())
        if pool_scale is not None:
            out = out * pool_scale.double().unsqueeze(1)
        pooled.copy_(out.float())


def relu_bn_bwd_reduce(z, scale, shift, mean, rstd, d_out, d_pooled, pool_scale, d_score, u, d_neg, n_neg,
                       node_off, n_graphs, dy, stats, tail=None):
    m, f = z.shape
    gid = _graph_of_row(node_off, m)
    g = torch.zeros(m, f, dtype=torch.float32)
    if d_out is not None:
        g = g + d_out
    if d_pooled is not None:
        gp = d_pooled if pool_scale is None else d_pooled * pool_scale.unsqueeze(1)
        g = g + gp[gid]
    if d_score is not None:
        g = g + d_score.reshape(-1, 1) * u[gid]
    if d_neg is not None and n_neg > 0:
        k = min(n_neg, m)
        g[:k] = g[:k] + d_neg[:k]
    v = torch.where(z * scale + shift > 0, g, torch.zeros_like(g))
    dy.copy_(v)
    if stats is not None:
        stats[:f] += v.double().sum(0)
        stats[f:] += (v.double() * ((z - mean) * rstd).double()).sum(0)


def bn_bwd_apply(z, mean, rstd, gamma, stats, count, dy):
    f = dy.shape[1]
    v = dy
    if stats is not None:
        m1 = (stats[:f] / count).float()
        m2 = (stats[f:] / count).float()
        v = v - m1 - (z - mean) * rstd * m2
    dy.copy_(v * gamma * rstd)


def gather_nf_rows(h_all, n_rows):
    return torch.cat([h_all[l, :n_rows] for l in range(h_all.shape[0])], 1).contiguous()


def dgi_score_fwd(h_all, u, neg_table, neg_idx, node_off, n_graphs, bias, out):
    m = h_all.shape[1]
    gid = _graph_of_row(node_off, m)
    nf = torch.cat([h_all[l] for l in range(h_all.shape[0])], 1)
    flat = out.view(-1)
    flat[:m] = (nf * u[gid]).sum(1) + bias
    s2 = (neg_table[neg_idx.long()] * u).sum(1) + bias
    flat[m:] = s2[gid]
    return out


def dgi_score_bwd(h_all, d_out, neg_table, neg_idx, node_off, n_graphs, du, s2, d_bias):
    m = h_all.shape[1]
    gid = _graph_of_row(node_off, m)
    nf = torch.cat([h_all[l] for l in range(h_all.shape[0])], 1)
    d1, d2 = d_out[:m], d_out[m:]
    s = torch.zeros(n_graphs).index_add_(0, gid, d2)
    s2.copy_(s)
    acc = torch.zeros(n_graphs, nf.shape[1]).index_add_(0, gid, d1.unsqueeze(1) * nf)
    du.copy_(acc + s.unsqueeze(1) * neg_table[neg_idx.long()])
    if d_bias is not None:
        d_bias += d_out.double().sum()


def rowdot_score(h, u, rows_per_graph, bias, s_bias, out):
    gid = torch.arange(h.shape[0]) // rows_per_graph
    v = (h * u[gid]).sum(1) + bias
    if s_bias is not None:
        v = v + s_bias.view(-1)
    out.copy_(v)
    return out


# ---- the [B, L*F]-sized remainder of a training step (contract of gnm_train.cu) ---------------

def small_gemm(a, a_strides, b, b_strides, c, m, n, k, sigmoid_a_out=None, dsig_s=None, dsig_add=None):
    am = torch.as_strided(a, (m, k), (int(a_strides[0]), int(a_strides[1]))).double()
    bm = torch.as_strided(b, (k, n), (int(b_strides[0]), int(b_strides[1]))).double()
    if sigmoid_a_out is not None:
        am = torch.sigmoid(am)
        sigmoid_a_out.copy_(am.to(sigmoid_a_out.dtype))
    out = am @ bm
    if dsig_s is not None:
        s = dsig_s.double()
        out = out * s * (1.0 - s)
        if dsig_add is not None:
            out = out + dsig_add.double()
    c.copy_(out.to(c.dtype))
    return c


def dgi_neg_grad(neg_idx, s2, u, d_neg):
    d_neg.zero_()
    d_neg.index_add_(0, neg_idx.long(), s2.unsqueeze(1) * u)
    return d_neg


def aggregate_dense_table(bitmap_addr, node_off, rowptr, n_graphs, n_max, table, tags, dst, mode, eps, bias, out_stats, tail=None):
    return False          # the stand-in has no shared-table kernel: the engine falls back to aggregate + col_stats


# ---- attribution (contracts of gnm_segment.cu, gnm_ig.cu, gnm_occlusion.cu) --------------------

def segment_weighted_colsum(x, node_off, out, z=None, coef=None, rowptr=None, mode=0, eps=None):
    """gnm_segment_weighted_colsum: out[g] = (1/n_g) sum_{m in g} w_m v[m], v = x or cA x + cB z + cC, w_m the row sums
    of the aggregation operator (deg, or 1 / 0 for an isolated node under average, + 1 + eps), zeros for an empty graph."""
    v = x.double()
    if coef is not None:
        v = coef[0].double() * v
        if z is not None:
            v = v + coef[1].double() * z.double() + coef[2].double()
    m = x.shape[0]
    if rowptr is None:
        w = torch.ones(m, dtype=torch.float64)
    else:
        deg = (rowptr[1:] - rowptr[:-1]).double()
        w = (deg > 0).double() if mode == 1 else deg
        if eps is not None:
            w = w + 1.0 + eps.double()
    no = node_off.long()
    gid = torch.repeat_interleave(torch.arange(no.numel() - 1), no[1:] - no[:-1])
    s = torch.zeros(out.shape[0], x.shape[1], dtype=torch.float64).index_add_(0, gid, w.unsqueeze(1) * v)
    n = (no[1:] - no[:-1]).double().clamp(min=1).unsqueeze(1)
    out.copy_((s / n).float())
    return out


def ig_expand(p, bias, alpha, node_off, points, z):
    """gnm_ig_expand: z[(g, s, i)] = alpha[s] * p[node_off[g] + i] + bias, graph-major virtual rows."""
    no = node_off.long().tolist()
    rows = []
    for g in range(len(no) - 1):
        for s in range(points):
            v = float(alpha[s]) * p[no[g]:no[g + 1]].double()
            rows.append(v + bias.double() if bias is not None else v)
    if rows:
        z.copy_(torch.cat(rows).float())
    return z


def ig_accumulate(dy, coef, node_off, points, weight, out, accumulate):
    """gnm_ig_accumulate: out[r] (+)= weight * cA o sum_s dy[(g, s, r - node_off[g])]."""
    no = node_off.long().tolist()
    ca = coef[0].double() if coef is not None else 1.0
    for g in range(len(no) - 1):
        n = no[g + 1] - no[g]
        base = points * no[g]
        v = weight * ca * dy[base:base + points * n].double().view(points, n, -1).sum(0)
        if accumulate:
            v = v + out[no[g]:no[g + 1]].double()
        out[no[g]:no[g + 1]] = v.float()
    return out


def ig_attribute(t, table, tags, node_off, out):
    """gnm_ig_attribute: out[g, d] = (1/n_g) sum_{n in g, tags[n] = d} <t[n], table[d]>; NaN row for non-finite t."""
    a = (t.double() * table.double()[tags.long()]).sum(1)
    no = node_off.long().tolist()
    for g in range(len(no) - 1):
        r0, r1 = no[g], no[g + 1]
        row = torch.zeros(out.shape[1], dtype=torch.float64).index_add_(0, tags[r0:r1].long(), a[r0:r1])
        row = row / max(r1 - r0, 1)
        if not bool(torch.isfinite(t[r0:r1]).all()):
            row[:] = float("nan")
        out[g] = row.float()
    return out


def occlusion_expand(p, bias, w1t, rowptr, colidx, tags, node_off, n_max, v_graph, v_tag, v_node_off, mode, eps, z):
    """gnm_occlusion_expand: z[v_node_off[v] + i] = p[m] + bias - c_d[m] w1t[d], c_d[m] = s_m #{n in CSR row m:
    tags[n] = d} + (eps ? (1 + eps) [tags[m] = d] : 0), s_m = 1 (mode 0) or 1 / (row length) (mode 1)."""
    m_all = p.shape[0]
    rp, ci, tg = rowptr.long(), colidx.long(), tags.long()
    rows = torch.repeat_interleave(torch.arange(m_all), rp[1:] - rp[:-1])
    counts = torch.zeros(m_all, w1t.shape[0], dtype=torch.float64)
    counts.index_put_((rows, tg[ci]), torch.ones(ci.numel(), dtype=torch.float64), accumulate=True)
    deg = (rp[1:] - rp[:-1]).double()
    no, vno = node_off.long().tolist(), v_node_off.long().tolist()
    base = p.double() + (bias.double() if bias is not None else 0.0)
    for v in range(v_graph.shape[0]):
        g, d = int(v_graph[v]), int(v_tag[v])
        r0, r1 = no[g], no[g + 1]
        val = base[r0:r1].clone()
        if 0 <= d < w1t.shape[0]:
            c = counts[r0:r1, d]
            coef = torch.where(c != 0, c / deg[r0:r1] if mode == 1 else c, torch.zeros_like(c))
            if eps is not None:
                coef = coef + (1.0 + float(eps[0])) * (tg[r0:r1] == d).double()
            val = val - coef.unsqueeze(1) * w1t[d].double()
        z[vno[v]:vno[v] + r1 - r0] = val.float()
    return z
