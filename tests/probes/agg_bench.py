"""Micro-benchmark / ncu target for the neighbour-aggregation kernels at the benchmark shape
(B graphs x N nodes, F features): python tests/probes/agg_bench.py [B] [iters] [impl] [N] [F]"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from graph_neural_mapping_b200 import engine, ops, synth  # noqa: E402


def main():
    b = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    iters = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    impls = [int(x) for x in sys.argv[3:4]] or [2, 1, 0]
    n_nodes = int(sys.argv[4]) if len(sys.argv) > 4 else 400
    dev = torch.device("cuda")
    graphs = synth.make_graphs_bulk(b, n_nodes, 30, 128, seed0=0, device=dev)
    store = engine.GraphStore(dev, add_self_loops=True)
    bs = store.assemble(store.assemble_host(graphs), "sum")
    m, f = bs.n_rows, (int(sys.argv[5]) if len(sys.argv) > 5 else 64)
    torch.manual_seed(0)
    src = torch.randn(m, f, device=dev)
    dst = torch.empty(m, f, device=dev)
    ref = torch.empty(m, f, device=dev)
    ops.aggregate(bs.rowptr, bs.colidx, src, None, ref, 0, None, None)
    alg_bytes = 4.0 * bs.nnz + 4.0 * (m + 1) + 8.0 * m * f
    for impl in impls:
        if impl == 3:
            # the backward pass's fused variant: aggregation -> + readout / DGI gradients -> ReLU mask of the layer below ->
            # BatchNorm-backward sums, as the step calls it for the middle layers (no eps, no negative rows)
            z = torch.randn(m, f, device=dev)
            scale = torch.rand(f, device=dev) + 0.5
            shift = torch.randn(f, device=dev) * 0.1
            mean = torch.randn(f, device=dev) * 0.1
            rstd = torch.rand(f, device=dev) + 0.5
            d_pooled = torch.randn(bs.n_graphs, f, device=dev)
            d_score = torch.randn(m, device=dev)
            u = torch.randn(bs.n_graphs, f, device=dev)
            stats = torch.zeros(2, f, dtype=torch.float64, device=dev)
            # PROBE_STEP (bit mask): the extras of the training step's call, one by one: 1 = readout / DGI operands as
            # column slices of [B, 5F] matrices, 2 = negative-row gradients for the first B rows, 4 = pool scale,
            # 8 = BatchNorm-backward tail in the last CTA
            flags = int(os.environ.get("PROBE_STEP", "0"))
            d_neg, n_neg, ps, tail = None, 0, None, None
            if flags & 1:
                d_pooled = torch.randn(bs.n_graphs, 5 * f, device=dev)[:, f:2 * f]
                u = torch.randn(bs.n_graphs, 5 * f, device=dev)[:, f:2 * f]
            if flags & 2:
                d_neg, n_neg = torch.randn(bs.n_graphs, 5 * f, device=dev)[:, f:2 * f], bs.n_graphs
            if flags & 4:
                ps = torch.ones(bs.n_graphs, device=dev)
            if flags & 8:
                coef = torch.empty(3, f, device=dev)
                tail = ops.BnTail(ops.BnTail.BWD_COEFFS, float(m), scale, mean, rstd, coef=coef)
            fn = lambda: ops.aggregate_dense_relu_bn_bwd(bs.bitmap_addr, bs.node_off, bs.rowptr, bs.n_graphs, bs.n_max, src, 0,
                                                         None, z, scale, shift, mean, rstd, d_pooled, ps, d_score, u, d_neg, n_neg,
                                                         dst, stats, tail)
            name = "tcgen05 fused bwd"
        elif impl == 4:
            # layer 0: one 400 x F table shared by every graph (tags = arange), bias, BatchNorm statistics of the output
            table = torch.randn(n_nodes, f, device=dev)
            tags = torch.arange(n_nodes, dtype=torch.int32, device=dev)
            bias = torch.randn(f, device=dev)
            ostats = torch.zeros(2, f, dtype=torch.float64, device=dev)
            fn = lambda: ops.aggregate_dense_table(bs.bitmap_addr, bs.node_off, bs.rowptr, bs.n_graphs, bs.n_max, table, tags, dst,
                                                   0, None, bias, ostats)
            name = "tcgen05 table"
        elif impl == 5:
            # layer-0 backward: rows = cA * dy + cB * z + cC formed on load (two streams)
            z = torch.randn(m, f, device=dev)
            coef = torch.randn(3, f, device=dev)
            fn = lambda: ops.aggregate_dense_affine(bs.bitmap_addr, bs.node_off, bs.rowptr, bs.n_graphs, bs.n_max, src, z, coef, dst, 0)
            name = "tcgen05 affine"
        elif impl == 0:
            fn = lambda: ops.aggregate(bs.rowptr, bs.colidx, src, None, dst, 0, None, None)
            name = "csr warp-per-row"
        else:
            fn = lambda: ops.aggregate_dense(bs.bitmap_addr, bs.node_off, bs.rowptr, bs.n_graphs, bs.n_max, src, None, dst, 0,
                                             None, None, impl=impl)
            name = "mma.sync dense" if impl == 1 else "tcgen05 dense"
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
        ev[0].record()
        for i in range(iters):
            fn()
            ev[i + 1].record()
        torch.cuda.synchronize()
        ts = [ev[i].elapsed_time(ev[i + 1]) * 1e3 for i in range(iters)]
        if impl >= 2:
            from graph_neural_mapping_b200 import lib
            dbg = torch.zeros(148 * 16, dtype=torch.int64, device=dev)
            lib.load().gnm_aggregate_tc_set_debug(dbg.data_ptr())
            fn()
            torch.cuda.synchronize()
            lib.load().gnm_aggregate_tc_set_debug(None)
            d = dbg.view(148, 16).double().mean(0).tolist()
            print("  tcgen05 role cycles (mean over CTAs): epilogue %.0f (waiting acc_full %.0f) | mma %.0f (waiting a_full %.0f, "
                  "acc_empty %.0f) | producer %.0f (a_empty slow-path wait %.0f; A expand+store %.0f, a_empty wait call incl. fast path %.0f, syncwarp+arrive %.0f, B convert+store+next loads %.0f, tile head/tail (word loads, item switch) %.0f) | epilogue warp 0: drain %.0f, copy-out %.0f" % tuple(d[:14]))
        if impl in (4, 5):
            if impl == 4:
                ops.aggregate(bs.rowptr, bs.colidx, table.repeat(bs.n_graphs, 1), None, ref, 0, None, None)
                want, alg = ref + bias, alg_bytes - 4.0 * m * f
            else:
                ops.aggregate(bs.rowptr, bs.colidx, coef[0] * src + coef[1] * z + coef[2], None, ref, 0, None, None)
                want, alg = ref, alg_bytes + 4.0 * m * f
            err = float((dst - want).abs().max() / want.abs().max())
            t = float(np.median(ts))
            print("%-18s median %8.1f us  min %8.1f us  -> %7.1f GB/s algorithmic (%.3f of 6546)  max rel err %.2e  abort=%s"
                  % (name, t, min(ts), alg / t / 1e3, alg / t / 1e3 / 6546.2, err, ops.aggregate_tc_status()))
            continue
        if impl == 3:
            want = ref + d_pooled.repeat_interleave(n_nodes, 0) + d_score[:, None] * u.repeat_interleave(n_nodes, 0)
            if d_neg is not None:
                want[:n_neg] += d_neg
            want = torch.where(z * scale + shift > 0, want, torch.zeros_like(want))
            err = float((dst - want).abs().max() / want.abs().max())
            alg = alg_bytes + 4.0 * m * f
            t = float(np.median(ts))
            print("%-18s median %8.1f us  min %8.1f us  -> %7.1f GB/s algorithmic (%.3f of 6546)  max rel err %.2e  abort=%s"
                  % (name, t, min(ts), alg / t / 1e3, alg / t / 1e3 / 6546.2, err, ops.aggregate_tc_status()))
            continue
        err = float((dst - ref).abs().max() / ref.abs().max())
        t = float(np.median(ts))
        print("%-18s median %8.1f us  min %8.1f us  -> %7.1f GB/s algorithmic (%.3f of 6546)  max rel err vs csr %.2e  abort=%s"
              % (name, t, min(ts), alg_bytes / t / 1e3, alg_bytes / t / 1e3 / 6546.2, err, ops.aggregate_tc_status()))


if __name__ == "__main__":
    main()
