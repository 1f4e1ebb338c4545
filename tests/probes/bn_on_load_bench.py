"""Micro-benchmark of BatchNorm + ReLU on load at the benchmark shape (B graphs x N nodes, F = 64): the tcgen05
aggregation reading the pre-BatchNorm z without / with the graph pooling, against the plain variant on a materialised h
and against bn_relu_readout with and without writing h; and the DGI / gather kernels with and without the scale | shift
table. CUDA events around each launch, median over the iterations; every [M, F] operand is 105 MB, larger than L2.
    python tests/probes/bn_on_load_bench.py [B] [iters] [N] [L]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from graph_neural_mapping_b200 import engine, ops, synth  # noqa: E402


def median_us(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(iters):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(200000)            # keep the device busy while the host records the start event
        s.record()
        fn()
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e) * 1e3)
    times.sort()
    return times[len(times) // 2]


def main():
    b = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    iters = int(sys.argv[2]) if len(sys.argv) > 2 else 30
    n = int(sys.argv[3]) if len(sys.argv) > 3 else 400
    L = int(sys.argv[4]) if len(sys.argv) > 4 else 5
    f = 64
    dev = torch.device("cuda")
    graphs = synth.make_graphs_bulk(b, n, 30, 128, seed0=0, device=dev)
    store = engine.GraphStore(dev, add_self_loops=True)
    bs = store.assemble(store.assemble_host(graphs), "sum")
    m = bs.n_rows
    torch.manual_seed(0)
    z = torch.randn(m, f, device=dev)
    scale = torch.rand(f, device=dev) + 0.5
    shift = torch.randn(f, device=dev) * 0.5
    ps = torch.full((b,), 1.0 / n, device=dev)
    h = torch.empty(m, f, device=dev)
    dst = torch.empty(m, f, device=dev)
    ref = torch.empty(m, f, device=dev)
    g_f = torch.empty(b, L * f, device=dev)
    g_ref = torch.empty(b, f, device=dev)
    agg = lambda src, out, **k: ops.aggregate_dense(bs.bitmap_addr, bs.node_off, bs.rowptr, b, bs.n_max, src, None, out, 0,
                                                    None, None, **k)
    ops.bn_relu_readout(z, scale, shift, h, bs.node_off, b, ps, g_ref)
    agg(h, ref, impl=2)
    calls = {
        "aggregate plain (materialised h)": lambda: agg(h, ref, impl=2),
        "aggregate bn on load": lambda: agg(z, dst, bn_scale=scale, bn_shift=shift),
        "aggregate bn on load + pooling": lambda: agg(z, dst, bn_scale=scale, bn_shift=shift, pooled=g_f[:, f:2 * f],
                                                      pool_scale=ps),
        "readout writing h": lambda: ops.bn_relu_readout(z, scale, shift, h, bs.node_off, b, ps, g_ref),
        "readout, pooling only": lambda: ops.bn_relu_readout(z, scale, shift, None, bs.node_off, b, ps, g_ref),
    }
    print("device: %s, B=%d N=%d L=%d F=%d" % (torch.cuda.get_device_name(), b, n, L, f))
    res = {k: median_us(fn, iters) for k, fn in calls.items()}
    same = bool(torch.equal(dst, ref))
    perr = float((g_f[:, f:2 * f] - g_ref).abs().max() / g_ref.abs().max())
    for k, v in res.items():
        print("%-34s %8.1f us" % (k, v))
    print("on-load output equal to readout -> aggregate: %s, pooled max rel err %.2e, abort=%s"
          % (same, perr, ops.aggregate_tc_status()))
    print("per step, L-1 aggregations + readouts: pooling in the aggregation %.1f us, read-only readout per layer %.1f us, "
          "materialised h %.1f us" % ((L - 1) * res["aggregate bn on load + pooling"] + res["readout, pooling only"],
                                     (L - 1) * res["aggregate bn on load"] + L * res["readout, pooling only"],
                                     (L - 1) * res["aggregate plain (materialised h)"] + L * res["readout writing h"]))

    # DGI / gather: the L slices of z with the [L, 2, F] scale | shift table against materialised h
    del h, dst, ref
    zl = torch.randn(L, m, f, device=dev)
    hl = torch.empty(L, m, f, device=dev)
    bn = torch.rand(L, 2, f, device=dev) + 0.5
    u = 0.2 * torch.randn(b, L * f, device=dev)
    bias = torch.tensor([0.3], device=dev)
    perm = torch.randperm(b, device=dev).to(torch.int32)
    no = bs.node_off
    table = ops.gather_nf_rows(zl, b, bn=bn)
    w = 0.05 / (2.0 * m)
    out = torch.empty(2 * m, 1, device=dev)
    dd = torch.randn(2 * m, device=dev)
    ds = torch.empty(m, device=dev)
    du, s2 = torch.empty(b, L * f, device=dev), torch.empty(b, device=dev)
    db, loss = torch.zeros(1, dtype=torch.float64, device=dev), torch.zeros(1, dtype=torch.float64, device=dev)
    dgi = {}
    for tag, src, bnt in (("", hl, None), ("+bn", zl, bn)):
        k = {"bn": bnt} if bnt is not None else {}
        dgi["gather_nf_rows" + tag] = lambda src=src, k=k: ops.gather_nf_rows(src, b, out=table, **k)
        dgi["dgi_score_fwd" + tag] = lambda src=src, k=k: ops.dgi_score_fwd(src, u, table, perm, no, b, bias, out, **k)
        dgi["dgi_score_bwd" + tag] = lambda src=src, k=k: ops.dgi_score_bwd(src, dd, table, perm, no, b, du, s2, db, **k)
        dgi["dgi_score_train" + tag] = lambda src=src, k=k: ops.dgi_score_train(src, u, table, perm, no, b, bias, w, w, out,
                                                                              ds, du, s2, db, loss, **k)
    for k, fn in dgi.items():
        print("%-34s %8.1f us" % (k, median_us(fn, iters)))


if __name__ == "__main__":
    main()
