"""ROI occlusion against the composed route of existing code at the benchmark shape (B graphs x N nodes, D = N one-hot
inputs, F = 64, 5 layers, sum / sum, eval, classes 0 and 1, occlusions_per_pass = 1024). Prints the GPU name, power
limit and max SM clock, then medians of CUDA-event timings after warm-up:
  1. compute_roi_occlusion_batched(classes=(0, 1)) including the D2H copy of its [B, 2, D] result;
  2. the composed route: per ROI d, driver.class_logits on dense copies of the B graphs with column d set to 0. Only
     `composed_rois` ROIs are timed, alternating with (1); the per-ROI median is scaled by D (every ROI costs the same),
     and one class_logits call on the unoccluded graphs is added once;
  3. gnm_occlusion_expand alone on one pass (occlusions_per_pass virtual graphs), with the achieved rate on its
     algorithmic bytes and its fraction of the 6546 GB/s copy peak DESIGN.md section 4 uses;
  4. (1) under max neighbour pooling at B_max graphs, labelled as such.
Successive timed calls cycle through `pools` disjoint graph sets (and the kernel through as many output buffers), so
that no call finds its inputs in the 126 MB L2.
    python tests/probes/roi_occlusion_bench.py [B] [iters] [pools] [composed_rois] [B_max]"""
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from graph_neural_mapping_b200 import driver, ops, synth  # noqa: E402
from graph_neural_mapping_b200.models import GIN_InfoMaxReg  # noqa: E402
from graph_neural_mapping_b200.models.graphcnn import occlusion_passes  # noqa: E402
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


def make_model(d, f, neigh, dev):
    torch.manual_seed(0)
    model = GIN_InfoMaxReg(5, 2, d, f, 2, 0.0, False, "sum", neigh, dev).to(dev)
    model.eval()
    return model


def main():
    b = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
    iters = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    pools = int(sys.argv[3]) if len(sys.argv) > 3 else 3
    composed_rois = int(sys.argv[4]) if len(sys.argv) > 4 else 3
    b_max = int(sys.argv[5]) if len(sys.argv) > 5 else 64
    n, f, opp = 400, 64, 1024
    d = n
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv"],
                         stdout=subprocess.PIPE, text=True).stdout.strip())
    dev = torch.device("cuda")
    model = make_model(d, f, "sum", dev)
    sets = [synth.make_graphs_bulk(b, n, 30, 128, seed0=1000 * k, device=dev) for k in range(pools)]
    host = torch.empty(b * 2 * d, dtype=torch.float32, pin_memory=True)

    def call(k, m=model, s=sets):
        r = m.compute_roi_occlusion_batched(s[k], (0, 1), occlusions_per_pass=opp)
        host[:r.numel()].copy_(r.reshape(-1), non_blocking=True)

    # the composed route's inputs: dense copies with one column zeroed (built outside the timed window), one ROI per pool
    rois = np.random.default_rng(0).choice(d, size=pools, replace=False).tolist()
    copies = []
    for k in range(pools):
        cs = []
        for g in sets[k]:
            x = g.node_features.to(dev, torch.float32).clone()
            x[:, rois[k]] = 0
            cs.append(SynthGraph(n, g.label, g.edge_mat, x))
        copies.append(cs)

    def composed_roi(k):
        driver.class_logits(model, copies[k], batch=b)

    for i in range(2 * pools):
        call(i % pools)
        composed_roi(i % pools)
    torch.cuda.synchronize()
    t_call, t_roi = [], []
    for i in range(max(iters, composed_rois)):
        if i < iters:
            t_call.append(timed(call, i % pools))
        if i < composed_rois:
            t_roi.append(timed(composed_roi, i % pools))
    t_call, t_roi = stats(t_call), stats(t_roi)
    t_base = median_ms(lambda k: driver.class_logits(model, sets[k], batch=b), iters, pools)

    # the kernel alone, at the first pass of the call above
    h = model._host_batch(sets[0])
    rbs = model._structure(sets[0], h)
    v_graph, v_tag = occlusion_passes(h.node_off, rbs.tags.cpu().numpy(), opp)[0]
    real = sorted(set(v_graph.tolist()))
    vbs = model._structure([sets[0][g] for g in v_graph.tolist()])
    m_v, m_r = vbs.n_rows, len(real) * n
    p0 = torch.randn(rbs.n_rows, f, device=dev)
    w1t = torch.randn(d, f, device=dev)
    bias = torch.randn(f, device=dev)
    vg, vt = torch.from_numpy(v_graph).to(dev), torch.from_numpy(v_tag).to(dev)
    zs = [torch.empty(m_v, f, device=dev) for _ in range(pools)]
    colidx = rbs.colidx
    t_exp = median_ms(lambda k: ops.occlusion_expand(p0, bias, w1t, rbs.rowptr, colidx, rbs.tags, rbs.node_off, rbs.n_max,
                                                     vg, vt, vbs.node_off, 0, None, zs[k]), 20 * iters, pools)
    # written rows, read P rows of the pass's real graphs, their tags, the CSR rows of the occluded nodes (one node per
    # tag here), the W1 rows, and the virtual-graph tables
    deg = (rbs.rowptr[1:] - rbs.rowptr[:-1]).double().mean().item()
    n_occ = int((v_tag >= 0).sum())
    by_exp = int(4 * m_v * f + 4 * m_r * f + 4 * m_r + n_occ * (8 + 4 * deg) + 4 * n_occ * f + 12 * len(v_graph))

    # max neighbour pooling: a smaller B, the layers above 0 on the CSR gather kernels
    model_max = make_model(d, f, "max", dev)
    sets_max = [s[:b_max] for s in sets]
    t_max = median_ms(lambda k: call(k, model_max, sets_max), iters, pools)

    n_pass = len(occlusion_passes(h.node_off, rbs.tags.cpu().numpy(), opp))
    print("shape: B = %d graphs x N = %d nodes, D = %d, F = %d, 5 layers, classes 0 and 1, occlusions_per_pass = %d "
          "(%d passes); %d disjoint graph sets cycled" % (b, n, d, f, opp, n_pass, pools))
    print("%-58s median %9.2f ms (min %.2f, max %.2f)  %7.3f k graphs/s" % (
        "1. compute_roi_occlusion_batched + D2H", t_call[0], t_call[1], t_call[2], b / t_call[0]))
    composed = t_roi[0] * d + t_base[0]
    print("%-58s median %9.2f ms (min %.2f, max %.2f) per ROI, x %d + %.2f ms unoccluded = %.1f ms  %7.3f k graphs/s" % (
        "2. composed route (class_logits on dense copies)", t_roi[0], t_roi[1], t_roi[2], d, t_base[0], composed,
        b / composed))
    print("   speed-up of (1) over (2): %.1fx" % (composed / t_call[0]))
    rate = by_exp / (t_exp[0] * 1e-3)
    print("%-58s median %9.1f us (min %.1f, max %.1f)  %.0f GB/s on %.1f MB = %.2f of copy peak" % (
        "3. occlusion_expand alone (one pass, %d virtual graphs)" % len(v_graph), t_exp[0] * 1e3, t_exp[1] * 1e3,
        t_exp[2] * 1e3, rate / 1e9, by_exp / 1e6, rate / COPY_PEAK))
    print("%-58s median %9.2f ms (min %.2f, max %.2f)  %7.3f k graphs/s" % (
        "4. MAX neighbour pooling, B = %d: call + D2H" % b_max, t_max[0], t_max[1], t_max[2], b_max / t_max[0]))


if __name__ == "__main__":
    main()
