// Per-graph weighted column sums (include/gnm.h: gnm_segment_weighted_colsum): the node average of the saliency maps
// without the maps. One CTA per (graph, column tile) streams the graph's rows once; each thread owns one vector column
// and a fixed residue class of rows, and the row groups are combined in shared memory in a fixed order, so the result
// is deterministic and no atomics touch the output.
#include "gnm_common.cuh"

namespace {

constexpr int SC_THREADS = 128;
constexpr int SC_UNROLL = 4;       // rows in flight per thread

struct SegColsumP {
    const float* x; int64_t ldx;
    const float* z; int64_t ldz;
    const float* coef;             // [cA | cB | cC], width each; nullable
    const int32_t* node_off;
    const int32_t* rowptr;         // nullable: unit weights
    const float* eps;              // nullable: no self term
    float* out; int64_t ld_out;
    int width, mode;
};

template <int V>
__device__ __forceinline__ void load_row(const float* p, float (&r)[V]) {
    if constexpr (V == 4) {
        const float4 t = __ldcs(reinterpret_cast<const float4*>(p));
        r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
    } else {
        r[0] = __ldcs(p);
    }
}

// Row sum of the aggregation operator as its backward applies it (gnm_aggregate mode 0 sum / 2 transpose of the average,
// eps self term): deg, or 1 (0 for an isolated node, which no row gathers from) - plus 1 + eps.
__device__ __forceinline__ float row_weight(const SegColsumP& p, int r, float self_c) {
    if (p.rowptr == nullptr) return 1.f;
    const int deg = __ldg(p.rowptr + r + 1) - __ldg(p.rowptr + r);
    const float w = p.mode == 1 ? (deg > 0 ? 1.f : 0.f) : (float)deg;
    return p.eps != nullptr ? w + self_c : w;
}

template <int V, bool kAff, bool kZ>
__global__ void __launch_bounds__(SC_THREADS)
segment_weighted_colsum_kernel(const SegColsumP p, int tpr_log2) {
    __shared__ float red[SC_THREADS * V];
    const int g = blockIdx.x;
    const int tpr = 1 << tpr_log2, n_groups = SC_THREADS >> tpr_log2;
    const int lc = threadIdx.x & (tpr - 1), grp = threadIdx.x >> tpr_log2;
    const int col = (blockIdx.y * tpr + lc) * V;
    const bool col_ok = col < p.width;
    const int r0 = __ldg(p.node_off + g), r1 = __ldg(p.node_off + g + 1);
    float acc[V], ca[V], cb[V], cc[V];
#pragma unroll
    for (int k = 0; k < V; ++k) { acc[k] = 0.f; ca[k] = 1.f; cb[k] = 0.f; cc[k] = 0.f; }
    if (col_ok) {
        if (kAff) {
#pragma unroll
            for (int k = 0; k < V; ++k) {
                ca[k] = __ldg(p.coef + col + k);
                if (kZ) { cb[k] = __ldg(p.coef + p.width + col + k); cc[k] = __ldg(p.coef + 2 * p.width + col + k); }
            }
        }
        const float self_c = p.eps != nullptr ? 1.f + __ldg(p.eps) : 0.f;
        auto add_row = [&](const float (&xv)[V], const float (&zv)[V], float w) {
#pragma unroll
            for (int k = 0; k < V; ++k) {
                const float v = !kAff ? xv[k] : kZ ? fmaf(ca[k], xv[k], fmaf(cb[k], zv[k], cc[k])) : ca[k] * xv[k];
                acc[k] = fmaf(w, v, acc[k]);
            }
        };
        int r = r0 + grp;
        for (; r + (SC_UNROLL - 1) * n_groups < r1; r += SC_UNROLL * n_groups) {
            float xv[SC_UNROLL][V], zv[SC_UNROLL][V], w[SC_UNROLL];
#pragma unroll
            for (int u = 0; u < SC_UNROLL; ++u) {
                const int64_t rr = r + u * n_groups;
                load_row<V>(p.x + rr * p.ldx + col, xv[u]);
                if (kZ) load_row<V>(p.z + rr * p.ldz + col, zv[u]);
                w[u] = row_weight(p, (int)rr, self_c);
            }
#pragma unroll
            for (int u = 0; u < SC_UNROLL; ++u) add_row(xv[u], zv[u], w[u]);
        }
        for (; r < r1; r += n_groups) {
            float xv[V], zv[V];
            load_row<V>(p.x + (int64_t)r * p.ldx + col, xv);
            if (kZ) load_row<V>(p.z + (int64_t)r * p.ldz + col, zv);
            add_row(xv, zv, row_weight(p, r, self_c));
        }
    }
    // fixed-order combine of the row groups: group 0 adds groups 1, 2, ... in turn
#pragma unroll
    for (int k = 0; k < V; ++k) red[threadIdx.x * V + k] = acc[k];
    __syncthreads();
    if (grp != 0 || !col_ok) return;
    const int n = r1 - r0;
    const float scale = n > 0 ? 1.f / (float)n : 0.f;
#pragma unroll
    for (int k = 0; k < V; ++k) {
        float s = acc[k];
        for (int j = 1; j < n_groups; ++j) s += red[(j * tpr + lc) * V + k];
        if (col + k < p.width) p.out[(int64_t)g * p.ld_out + col + k] = s * scale;
    }
}

template <int V, bool kAff, bool kZ>
cudaError_t launch_colsum(const SegColsumP& p, int n_graphs, cudaStream_t st) {
    const int n_vec = (p.width + V - 1) / V;
    int tpr_log2 = 0;
    while ((1 << tpr_log2) < n_vec && (1 << tpr_log2) < SC_THREADS) ++tpr_log2;
    const dim3 grid(n_graphs, (n_vec + (1 << tpr_log2) - 1) >> tpr_log2);
    gnm_count_launch(GNM_K_SEGMENT_COLSUM);
    segment_weighted_colsum_kernel<V, kAff, kZ><<<grid, SC_THREADS, 0, st>>>(p, tpr_log2);
    return cudaGetLastError();
}

}  // namespace

extern "C" int gnm_segment_weighted_colsum(const float* x, int64_t ldx, const float* z, int64_t ldz, const float* coef,
                                           const int32_t* node_off, int n_graphs, int width, const int32_t* rowptr,
                                           int mode, const float* eps, float* out, int64_t ld_out, gnm_stream_t stream) {
    if (n_graphs < 0 || width < 0 || mode < 0 || mode > 1) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || width == 0) return GNM_OK;
    if (!x || !node_off || !out || (z != nullptr && coef == nullptr)) return GNM_ERR_BAD_ARG;
    if (ldx < width || ld_out < width || (z != nullptr && ldz < width)) return GNM_ERR_BAD_ARG;
    const SegColsumP p{x, ldx, z, ldz, coef, node_off, rowptr, eps, out, ld_out, width, mode};
    const bool vec4 = (width % 4 == 0) && (ldx % 4 == 0) && gnm_aligned16(x) &&
                      (z == nullptr || ((ldz % 4 == 0) && gnm_aligned16(z)));
    cudaStream_t st = gnm_cast_stream(stream);
    cudaError_t e;
    if (vec4) {
        e = coef == nullptr ? launch_colsum<4, false, false>(p, n_graphs, st)
          : z == nullptr    ? launch_colsum<4, true, false>(p, n_graphs, st)
                            : launch_colsum<4, true, true>(p, n_graphs, st);
    } else {
        e = coef == nullptr ? launch_colsum<1, false, false>(p, n_graphs, st)
          : z == nullptr    ? launch_colsum<1, true, false>(p, n_graphs, st)
                            : launch_colsum<1, true, true>(p, n_graphs, st);
    }
    return e == cudaSuccess ? GNM_OK : (int)e;
}
