"""Micro-benchmark of the DGI scoring kernels at the benchmark shape (B graphs x N nodes, L layers of F = 64): the
training step's one-pass scorer (gnm_dgi_score_train) against the three calls it replaces (gnm_dgi_score_fwd,
gnm_bce_logits, gnm_dgi_score_bwd). CUDA events around each launch, median over the iterations; n_f is 525 MB at the
default shape, so every launch streams it from HBM.
    python tests/probes/dgi_bench.py [B] [iters] [N] [L]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from graph_neural_mapping_b200 import ops  # noqa: E402


def median_us(fn, iters):
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
    iters = int(sys.argv[2]) if len(sys.argv) > 2 else 50
    n = int(sys.argv[3]) if len(sys.argv) > 3 else 400
    L = int(sys.argv[4]) if len(sys.argv) > 4 else 5
    f = 64
    dev = torch.device("cuda")
    m = b * n
    torch.manual_seed(0)
    h_all = torch.randn(L, m, f, device=dev)
    u = 0.2 * torch.randn(b, L * f, device=dev)
    bias = torch.tensor([0.3], device=dev)
    perm = torch.randperm(b, device=dev).to(torch.int32)
    no = torch.arange(0, m + 1, n, dtype=torch.int32, device=dev)
    table = ops.gather_nf_rows(h_all, b)
    w = 0.05 / (2.0 * m)
    out = torch.empty(2 * m, 1, device=dev)
    dd = torch.empty(2 * m, device=dev)
    ds = torch.empty(m, device=dev)
    du, s2 = torch.empty(b, L * f, device=dev), torch.empty(b, device=dev)
    db, loss = torch.zeros(1, dtype=torch.float64, device=dev), torch.zeros(1, dtype=torch.float64, device=dev)
    calls = {
        "dgi_score_fwd": lambda: ops.dgi_score_fwd(h_all, u, table, perm, no, b, bias, out),
        "bce_logits": lambda: ops.bce_logits(out.view(-1), m, w, w, loss, dd),
        "dgi_score_bwd": lambda: ops.dgi_score_bwd(h_all, dd, table, perm, no, b, du, s2, db),
        "dgi_score_train": lambda: ops.dgi_score_train(h_all, u, table, perm, no, b, bias, w, w, out, ds, du, s2, db, loss),
    }
    for fn in calls.values():
        for _ in range(5):
            fn()
    torch.cuda.synchronize()
    nf_bytes = 4.0 * L * m * f
    res = {k: median_us(fn, iters) for k, fn in calls.items()}
    three = res["dgi_score_fwd"] + res["bce_logits"] + res["dgi_score_bwd"]
    print("device: %s, B=%d N=%d L=%d F=%d, n_f = %.1f MB" % (torch.cuda.get_device_name(), b, n, L, f, nf_bytes / 1e6))
    for k, v in res.items():
        print("%-16s %8.1f us" % (k, v))
    print("three calls      %8.1f us   one pass %8.1f us   (%.2f TB/s of n_f in the one pass)"
          % (three, res["dgi_score_train"], nf_bytes / (res["dgi_score_train"] * 1e-6) / 1e12))


if __name__ == "__main__":
    main()
