"""ROI saliency against the full saliency maps at the benchmark shape (B graphs x N nodes, D = N one-hot inputs, F = 64,
5 layers, sum / sum, eval). Prints the GPU name and power limit, then medians of CUDA-event timings after warm-up:
  1. compute_saliency_batched for classes 0 and 1 (two calls), on the device;
  2. the same plus the D2H copy of both [M, D] maps into pinned host memory;
  3. compute_roi_saliency_batched(classes=(0, 1)) including the D2H copy of its [B, 2, D] result;
  4. gnm_segment_weighted_colsum alone on an [M, F] dy with the affine on load (eval: z not read) and the degree
     weights, with its achieved rate on the algorithmic bytes 4MF + 4(M+1) + 4BF.
Successive timed calls cycle through `pools` disjoint graph sets (and the kernel through as many dy buffers), so that
no call finds its inputs in the 126 MB L2.
    python tests/probes/roi_saliency_bench.py [B] [iters] [N] [pools]"""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from graph_neural_mapping_b200 import ops, synth  # noqa: E402
from graph_neural_mapping_b200.models import GIN_InfoMaxReg  # noqa: E402


def median_ms(fn, iters, pools):
    for i in range(2 * pools):
        fn(i % pools)
    torch.cuda.synchronize()
    times = []
    for i in range(iters):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn(i % pools)
        e.record()
        e.synchronize()
        times.append(s.elapsed_time(e))
    times.sort()
    return times[len(times) // 2], times[0], times[-1]


def main():
    b = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    iters = int(sys.argv[2]) if len(sys.argv) > 2 else 20
    n = int(sys.argv[3]) if len(sys.argv) > 3 else 400
    pools = int(sys.argv[4]) if len(sys.argv) > 4 else 3
    f, d = 64, n
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv"],
                         stdout=subprocess.PIPE, text=True).stdout.strip())
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = GIN_InfoMaxReg(5, 2, d, f, 2, 0.0, False, "sum", "sum", dev).to(dev)
    model.eval()
    sets = [synth.make_graphs_bulk(b, n, 30, 128, seed0=1000 * k, device=dev) for k in range(pools)]
    m = b * n
    pinned = [torch.empty(m * d, dtype=torch.float32, pin_memory=True) for _ in range(2)]
    roi_host = torch.empty(b * 2 * d, dtype=torch.float32, pin_memory=True)

    def full(k, copy=False):
        for c in (0, 1):
            s = model.compute_saliency_batched(sets[k], c)
            if copy:
                pinned[c].copy_(s.detach().reshape(-1), non_blocking=True)

    def roi(k):
        r = model.compute_roi_saliency_batched(sets[k], (0, 1))
        roi_host.copy_(r.reshape(-1), non_blocking=True)

    t_full = median_ms(lambda k: full(k), iters, pools)
    t_full_d2h = median_ms(lambda k: full(k, True), iters, pools)
    t_roi = median_ms(roi, iters, pools)

    # the kernel alone, on the batch structure of the first set
    bs = model._structure(sets[0])
    dys = [torch.randn(m, f, device=dev) for _ in range(pools)]
    coef = torch.randn(3, f, device=dev)
    out = torch.empty(b, f, device=dev)
    t_k = median_ms(lambda k: ops.segment_weighted_colsum(dys[k], bs.node_off, out, coef=coef, rowptr=bs.rowptr), 5 * iters,
                    pools)
    bytes_k = 4 * m * f + 4 * (m + 1) + 4 * b * f
    print("shape: B = %d graphs x N = %d nodes, D = %d, F = %d, 5 layers, 2 classes; %d disjoint graph sets cycled"
          % (b, n, d, f, pools))
    for name, t in (("1. compute_saliency_batched x2 (device)", t_full),
                    ("2. compute_saliency_batched x2 + D2H of both maps", t_full_d2h),
                    ("3. compute_roi_saliency_batched(0, 1) + D2H", t_roi)):
        print("%-52s median %8.3f ms (min %.3f, max %.3f)  %7.1f k graphs/s" % (name, t[0], t[1], t[2], b / t[0]))
    print("%-52s median %8.1f us (min %.1f, max %.1f)  %.0f GB/s on %.1f MB" % (
        "4. segment_weighted_colsum alone", t_k[0] * 1e3, t_k[1] * 1e3, t_k[2] * 1e3, bytes_k / (t_k[0] * 1e-3) / 1e9,
        bytes_k / 1e6))
    print("maps written per class: %.0f MB; ROI output per call: %.1f KB" % (m * d * 4 / 1e6, b * 2 * d * 4 / 1e3))


if __name__ == "__main__":
    main()
