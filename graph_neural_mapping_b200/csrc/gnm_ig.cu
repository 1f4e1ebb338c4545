// Integrated gradients on the one-hot layer 0 (include/gnm.h: gnm_ig_expand / gnm_ig_accumulate / gnm_ig_attribute).
// The path points of a chunk run as one virtual batch that repeats each real graph `points` times, graph-major; these
// kernels connect it to the real batch: layer 0's output at every point from one real-batch aggregation (expand), the
// quadrature sum of the points' layer-0 gradients (accumulate), and the per-ROI attribution (attribute). Every sum runs
// in a fixed order and no atomics touch an output, so a call is bit-reproducible.
#include "gnm_common.cuh"

namespace {

constexpr int IG_THREADS = 256;
constexpr int IG_UNROLL = 4;          // path points in flight per thread (accumulate)
constexpr int IG_TILE = 1024;         // nodes staged in shared memory per round (attribute)

// graph of real row r: the g with node_off[g] <= r < node_off[g+1] (empty graphs skipped)
__device__ __forceinline__ int graph_of_row(const int32_t* node_off, int n_graphs, int64_t r, int64_t scale) {
    int lo = 0, hi = n_graphs;        // invariant: scale*node_off[lo] <= r < scale*node_off[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (scale * (int64_t)__ldg(node_off + mid) <= r) lo = mid; else hi = mid;
    }
    return lo;
}

template <int V>
__device__ __forceinline__ void ld_vec(const float* p, float (&r)[V]) {
    if constexpr (V == 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p));
        r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
    } else {
        r[0] = __ldg(p);
    }
}

template <int V>
__device__ __forceinline__ void ld_vec_stream(const float* p, float (&r)[V]) {
    if constexpr (V == 4) {
        const float4 t = __ldcs(reinterpret_cast<const float4*>(p));
        r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
    } else {
        r[0] = __ldcs(p);
    }
}

template <int V>
__device__ __forceinline__ void st_vec(float* p, const float (&r)[V]) {
    if constexpr (V == 4) {
        *reinterpret_cast<float4*>(p) = make_float4(r[0], r[1], r[2], r[3]);
    } else {
        p[0] = r[0];
    }
}

// z[(g, s, i)] = alpha[s] * p[node_off[g] + i] + bias: one thread per (virtual row, vector column)
template <int V>
__global__ void __launch_bounds__(IG_THREADS)
ig_expand_kernel(const float* __restrict__ p, int64_t ldp, const float* __restrict__ bias,
                 const float* __restrict__ alpha, const int32_t* __restrict__ node_off, int n_graphs, int points,
                 int width, float* __restrict__ z, int64_t ldz, int64_t n_items) {
    const int n_vec = (width + V - 1) / V;
    for (int64_t it = (int64_t)blockIdx.x * IG_THREADS + threadIdx.x; it < n_items; it += (int64_t)gridDim.x * IG_THREADS) {
        const int64_t vr = it / n_vec;
        const int col = (int)(it - vr * n_vec) * V;
        const int g = graph_of_row(node_off, n_graphs, vr, points);
        const int64_t r0 = __ldg(node_off + g), n_g = __ldg(node_off + g + 1) - r0;
        const int64_t off = vr - points * r0;
        const int s = (int)(off / n_g);
        const int64_t r = r0 + (off - s * n_g);
        const float a = __ldg(alpha + s);
        float x[V], b[V], y[V];
        ld_vec<V>(p + r * ldp + col, x);
        if (bias != nullptr) ld_vec<V>(bias + col, b);
#pragma unroll
        for (int k = 0; k < V; ++k) y[k] = bias != nullptr ? fmaf(a, x[k], b[k]) : a * x[k];
        st_vec<V>(z + vr * ldz + col, y);
    }
}

// out[r] = (accumulate ? out[r] : 0) + weight * cA o sum_s dy[(g, s, r - node_off[g])]: one thread per (real row,
// vector column), the points summed in ascending order
template <int V>
__global__ void __launch_bounds__(IG_THREADS)
ig_accumulate_kernel(const float* __restrict__ dy, int64_t ldy, const float* __restrict__ coef,
                     const int32_t* __restrict__ node_off, int n_graphs, int points, int width, float weight,
                     int accumulate, float* __restrict__ out, int64_t ld_out, int64_t n_items) {
    const int n_vec = (width + V - 1) / V;
    for (int64_t it = (int64_t)blockIdx.x * IG_THREADS + threadIdx.x; it < n_items; it += (int64_t)gridDim.x * IG_THREADS) {
        const int64_t r = it / n_vec;
        const int col = (int)(it - r * n_vec) * V;
        const int g = graph_of_row(node_off, n_graphs, r, 1);
        const int64_t r0 = __ldg(node_off + g), n_g = __ldg(node_off + g + 1) - r0;
        const float* src = dy + (points * r0 + (r - r0)) * ldy + col;      // point 0 of row r
        const int64_t step = n_g * ldy;
        float acc[V];
#pragma unroll
        for (int k = 0; k < V; ++k) acc[k] = 0.f;
        int s = 0;
        for (; s + IG_UNROLL <= points; s += IG_UNROLL) {
            float v[IG_UNROLL][V];
#pragma unroll
            for (int u = 0; u < IG_UNROLL; ++u) ld_vec_stream<V>(src + (s + u) * step, v[u]);
#pragma unroll
            for (int u = 0; u < IG_UNROLL; ++u)
#pragma unroll
                for (int k = 0; k < V; ++k) acc[k] += v[u][k];
        }
        for (; s < points; ++s) {
            float v[V];
            ld_vec_stream<V>(src + s * step, v);
#pragma unroll
            for (int k = 0; k < V; ++k) acc[k] += v[k];
        }
        float ca[V], y[V];
        if (coef != nullptr) ld_vec<V>(coef + col, ca);
        else {
#pragma unroll
            for (int k = 0; k < V; ++k) ca[k] = 1.f;
        }
        float* dst = out + r * ld_out + col;
        if (accumulate) ld_vec<V>(dst, y);
#pragma unroll
        for (int k = 0; k < V; ++k) y[k] = accumulate ? fmaf(weight, ca[k] * acc[k], y[k]) : weight * (ca[k] * acc[k]);
        st_vec<V>(dst, y);
    }
}

// One CTA per graph. Per round of up to IG_TILE nodes: warp-per-node row dots a[n] = <t[n], table[tags[n]]> into
// shared memory, then thread c owns output columns c, c + IG_THREADS, ... and sums the a[n] whose tag is its column in
// node order (duplicate tags add up; no atomics). A non-finite entry in a row of t makes the graph's whole output NaN:
// the attribution X[n, d] * G[n, d] of every column d is 0 * non-finite there.
__global__ void __launch_bounds__(IG_THREADS)
ig_attribute_kernel(const float* __restrict__ t, int64_t ldt, const float* __restrict__ table, int64_t ld_table,
                    int n_table_rows, const int32_t* __restrict__ tags, const int32_t* __restrict__ node_off, int width,
                    float* __restrict__ out, int64_t ld_out) {
    __shared__ float a_sm[IG_TILE];
    __shared__ int tag_sm[IG_TILE];
    const int g = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int r0 = __ldg(node_off + g), r1 = __ldg(node_off + g + 1);
    float* o = out + (int64_t)g * ld_out;
    bool bad = false;
    for (int t0 = r0; t0 < r1; t0 += IG_TILE) {
        const int nt = min(IG_TILE, r1 - t0);
        __syncthreads();                       // the previous round's readers are done
        for (int i = warp; i < nt; i += IG_THREADS / 32) {
            const int64_t r = t0 + i;
            const int tag = __ldg(tags + r);
            const bool ok = tag >= 0 && tag < n_table_rows;
            const float* pt = t + r * ldt;
            const float* pw = table + (int64_t)(ok ? tag : 0) * ld_table;
            float acc = 0.f;
            for (int c = lane; c < width; c += 32) {
                const float v = __ldcs(pt + c);
                bad |= !isfinite(v);
                acc = fmaf(v, __ldg(pw + c), acc);
            }
            acc = warp_sum(acc);
            if (lane == 0) { a_sm[i] = acc; tag_sm[i] = ok ? tag : -1; }
        }
        __syncthreads();
        for (int d = threadIdx.x; d < n_table_rows; d += IG_THREADS) {
            float s = t0 == r0 ? 0.f : o[d];
            for (int i = 0; i < nt; ++i)
                if (tag_sm[i] == d) s += a_sm[i];
            o[d] = s;
        }
    }
    const bool any_bad = __syncthreads_or(bad);
    const int n = r1 - r0;
    const float scale = n > 0 ? 1.f / (float)n : 0.f;
    for (int d = threadIdx.x; d < n_table_rows; d += IG_THREADS)
        o[d] = any_bad ? __int_as_float(0x7fffffff) : (n > 0 ? o[d] * scale : 0.f);
}

int grid_for(int64_t n_items) {
    const int64_t b = (n_items + IG_THREADS - 1) / IG_THREADS;
    return (int)(b < 148 * 16 ? b : 148 * 16);
}

}  // namespace

extern "C" int gnm_ig_expand(const float* p, int64_t ldp, const float* bias, const float* alpha, const int32_t* node_off,
                             int n_graphs, int n_rows, int points, int width, float* z, int64_t ldz, gnm_stream_t stream) {
    if (n_graphs < 0 || n_rows < 0 || points < 0 || width < 0) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || n_rows == 0 || points == 0 || width == 0) return GNM_OK;
    if (!p || !alpha || !node_off || !z || ldp < width || ldz < width) return GNM_ERR_BAD_ARG;
    const bool vec4 = width % 4 == 0 && ldp % 4 == 0 && ldz % 4 == 0 && gnm_aligned16(p) && gnm_aligned16(z) &&
                      (bias == nullptr || gnm_aligned16(bias));
    const int v = vec4 ? 4 : 1;
    const int64_t n_items = (int64_t)points * n_rows * ((width + v - 1) / v);
    cudaStream_t st = gnm_cast_stream(stream);
    gnm_count_launch(GNM_K_IG_EXPAND);
    if (vec4)
        ig_expand_kernel<4><<<grid_for(n_items), IG_THREADS, 0, st>>>(p, ldp, bias, alpha, node_off, n_graphs, points,
                                                                       width, z, ldz, n_items);
    else
        ig_expand_kernel<1><<<grid_for(n_items), IG_THREADS, 0, st>>>(p, ldp, bias, alpha, node_off, n_graphs, points,
                                                                       width, z, ldz, n_items);
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}

extern "C" int gnm_ig_accumulate(const float* dy, int64_t ldy, const float* coef, const int32_t* node_off, int n_graphs,
                                 int n_rows, int points, int width, float weight, int accumulate, float* out,
                                 int64_t ld_out, gnm_stream_t stream) {
    if (n_graphs < 0 || n_rows < 0 || points < 0 || width < 0) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || n_rows == 0 || width == 0 || (points == 0 && accumulate)) return GNM_OK;
    if (!out || !node_off || ld_out < width || (points > 0 && (!dy || ldy < width))) return GNM_ERR_BAD_ARG;
    const bool vec4 = width % 4 == 0 && ldy % 4 == 0 && ld_out % 4 == 0 && (dy == nullptr || gnm_aligned16(dy)) &&
                      gnm_aligned16(out) && (coef == nullptr || gnm_aligned16(coef));
    const int v = vec4 ? 4 : 1;
    const int64_t n_items = (int64_t)n_rows * ((width + v - 1) / v);
    cudaStream_t st = gnm_cast_stream(stream);
    gnm_count_launch(GNM_K_IG_ACCUMULATE);
    if (vec4)
        ig_accumulate_kernel<4><<<grid_for(n_items), IG_THREADS, 0, st>>>(dy, ldy, coef, node_off, n_graphs, points,
                                                                           width, weight, accumulate, out, ld_out, n_items);
    else
        ig_accumulate_kernel<1><<<grid_for(n_items), IG_THREADS, 0, st>>>(dy, ldy, coef, node_off, n_graphs, points,
                                                                           width, weight, accumulate, out, ld_out, n_items);
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}

extern "C" int gnm_ig_attribute(const float* t, int64_t ldt, const float* table, int64_t ld_table, int n_table_rows,
                                const int32_t* tags, const int32_t* node_off, int n_graphs, int width, float* out,
                                int64_t ld_out, gnm_stream_t stream) {
    if (n_graphs < 0 || n_table_rows < 0 || width < 0) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || n_table_rows == 0) return GNM_OK;
    if (!node_off || !tags || !out || ld_out < n_table_rows) return GNM_ERR_BAD_ARG;
    if (width > 0 && (!t || !table || ldt < width || ld_table < width)) return GNM_ERR_BAD_ARG;
    gnm_count_launch(GNM_K_IG_ATTRIBUTE);
    ig_attribute_kernel<<<n_graphs, IG_THREADS, 0, gnm_cast_stream(stream)>>>(t, ldt, table, ld_table, n_table_rows, tags,
                                                                             node_off, width, out, ld_out);
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}
