"""Integrated gradients against the composed route of existing code at the benchmark shape (B graphs x N nodes, D = N
one-hot inputs, F = 64, 5 layers, sum / sum, eval, classes 0 and 1, `steps` path points). Prints the GPU name, power limit
and max SM clock, then medians of CUDA-event timings after warm-up:
  1. compute_integrated_gradients_batched(classes=(0, 1), steps) including the D2H copy of its [B, 2, D] result;
  2. the composed route: per path point, compute_saliency_batched for both classes on alpha-scaled dense copies of the
     graphs, times X, accumulated. Only `composed_points` points are timed, alternating with (1); the per-point median is
     scaled by `steps` (the points differ only in alpha, so each costs the same);
  3. gnm_ig_expand, gnm_ig_accumulate (one pass: B_pass = points_per_pass // steps graphs x steps points) and
     gnm_ig_attribute (B graphs) alone, with the achieved rate on their algorithmic bytes and its fraction of the
     6546 GB/s copy peak DESIGN.md section 4 uses.
Successive timed calls cycle through `pools` disjoint graph sets (and the kernels through as many input buffers), so that
no call finds its inputs in the 126 MB L2.
    python tests/probes/integrated_gradients_bench.py [B] [iters] [steps] [pools] [composed_points]"""
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from graph_neural_mapping_b200 import ops, synth  # noqa: E402
from graph_neural_mapping_b200.models import GIN_InfoMaxReg  # noqa: E402
from graph_neural_mapping_b200.synth import SynthGraph  # noqa: E402

COPY_PEAK = 6546e9


def timed(fn, arg):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    fn(arg)
    e.record()
    e.synchronize()
    return s.elapsed_time(e)


def stats(times):
    times = sorted(times)
    return times[len(times) // 2], times[0], times[-1]


def median_ms(fn, iters, pools):
    for i in range(2 * pools):
        fn(i % pools)
    torch.cuda.synchronize()
    return stats([timed(fn, i % pools) for i in range(iters)])


def main():
    b = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    iters = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    steps = int(sys.argv[3]) if len(sys.argv) > 3 else 50
    pools = int(sys.argv[4]) if len(sys.argv) > 4 else 3
    composed_points = int(sys.argv[5]) if len(sys.argv) > 5 else 3
    n, f, ppp = 400, 64, 1024
    d = n
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv"],
                         stdout=subprocess.PIPE, text=True).stdout.strip())
    dev = torch.device("cuda")
    torch.manual_seed(0)
    model = GIN_InfoMaxReg(5, 2, d, f, 2, 0.0, False, "sum", "sum", dev).to(dev)
    model.eval()
    sets = [synth.make_graphs_bulk(b, n, 30, 128, seed0=1000 * k, device=dev) for k in range(pools)]
    m = b * n
    ig_host = torch.empty(b * 2 * d, dtype=torch.float32, pin_memory=True)

    def ig(k):
        r = model.compute_integrated_gradients_batched(sets[k], (0, 1), steps=steps, points_per_pass=ppp)
        ig_host.copy_(r.reshape(-1), non_blocking=True)

    # the composed route's inputs: alpha-scaled dense copies (built outside the timed window), one alpha per pool
    xs = [torch.cat([g.node_features for g in sets[k]], 0).to(dev) for k in range(pools)]
    scaled = [[SynthGraph(n, g.label, g.edge_mat, ((k + 0.5) / steps) * g.node_features) for g in sets[k]]
              for k in range(pools)]
    acc = [torch.zeros(m, d, device=dev) for _ in range(2)]

    def composed_point(k):
        for c in (0, 1):
            acc[c] += xs[k] * model.compute_saliency_batched(scaled[k], c).detach()

    for i in range(2 * pools):
        ig(i % pools)
        composed_point(i % pools)
    torch.cuda.synchronize()
    t_ig, t_pt = [], []
    for i in range(max(iters, composed_points)):
        if i < iters:
            t_ig.append(timed(ig, i % pools))
        if i < composed_points:
            t_pt.append(timed(composed_point, i % pools))
    t_ig, t_pt = stats(t_ig), stats(t_pt)

    # the kernels alone, at one pass of the call above and on the first set's real batch
    per = max(1, ppp // steps)
    bs_all = model._structure(sets[0])
    bs_pass = model._structure(sets[0][:per])
    m_r, m_v = bs_pass.n_rows, bs_pass.n_rows * steps
    p0s = [torch.randn(m_r, f, device=dev) for _ in range(pools)]
    bias, alpha = torch.randn(f, device=dev), torch.rand(steps, device=dev)
    zs = [torch.empty(m_v, f, device=dev) for _ in range(pools)]
    t_exp = median_ms(lambda k: ops.ig_expand(p0s[k], bias, alpha, bs_pass.node_off, steps, zs[k]), 20 * iters, pools)
    coef = torch.randn(3, f, device=dev)
    acc_r = torch.empty(m_r, f, device=dev)
    t_acc = median_ms(lambda k: ops.ig_accumulate(zs[k], coef, bs_pass.node_off, steps, 1.0 / steps, acc_r, False),
                      20 * iters, pools)
    ts = [torch.randn(m, f, device=dev) for _ in range(pools)]
    table = torch.randn(d, f, device=dev)
    out = torch.empty(b, d, device=dev)
    t_att = median_ms(lambda k: ops.ig_attribute(ts[k], table, bs_all.tags, bs_all.node_off, out), 20 * iters, pools)
    by_exp = 4 * m_r * f + 4 * m_v * f + 4 * f + 4 * steps + 4 * (per + 1)
    by_acc = 4 * m_v * f + 4 * m_r * f + 4 * f + 4 * (per + 1)
    by_att = 4 * m * f + 4 * d * f + 4 * m + 4 * (b + 1) + 4 * b * d

    print("shape: B = %d graphs x N = %d nodes, D = %d, F = %d, 5 layers, classes 0 and 1, steps = %d, points_per_pass = %d "
          "(%d graphs x %d points per pass); %d disjoint graph sets cycled" % (b, n, d, f, steps, ppp, per, steps, pools))
    print("%-58s median %9.2f ms (min %.2f, max %.2f)  %7.2f k graphs/s" % (
        "1. compute_integrated_gradients_batched + D2H", t_ig[0], t_ig[1], t_ig[2], b / t_ig[0]))
    print("%-58s median %9.2f ms (min %.2f, max %.2f) per point, x %d = %.1f ms  %7.2f k graphs/s" % (
        "2. composed route (compute_saliency_batched x2 + X o grad)", t_pt[0], t_pt[1], t_pt[2], steps, t_pt[0] * steps,
        b / (t_pt[0] * steps)))
    print("   speed-up of (1) over (2): %.2fx" % (t_pt[0] * steps / t_ig[0]))
    for name, t, by in (("3a. ig_expand alone (one pass)", t_exp, by_exp), ("3b. ig_accumulate alone (one pass)", t_acc, by_acc),
                        ("3c. ig_attribute alone (B graphs)", t_att, by_att)):
        rate = by / (t[0] * 1e-3)
        print("%-58s median %9.1f us (min %.1f, max %.1f)  %.0f GB/s on %.1f MB = %.2f of copy peak" % (
            name, t[0] * 1e3, t[1] * 1e3, t[2] * 1e3, rate / 1e9, by / 1e6, rate / COPY_PEAK))


if __name__ == "__main__":
    main()
