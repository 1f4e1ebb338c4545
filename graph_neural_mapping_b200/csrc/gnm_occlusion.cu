// ROI occlusion on the one-hot layer 0 (include/gnm.h: gnm_occlusion_expand). Zeroing input column d changes layer 0's
// first Linear output by a rank-1 term, so every occluded copy of a graph is written from the real batch's
// p = Agg(X) W1^T: z[m] = p[m] + bias - c_d[m] * W1^T[d]. One CTA per virtual graph: the occurrence counts of tag d in
// each CSR row are integer shared-memory adds (exact in any order), then one pass writes every row of the copy once.
// No atomics touch z, so a call is bit-reproducible.
#include "gnm_common.cuh"

namespace {

constexpr int OC_THREADS = 256;
constexpr int OC_MAX_NODES = 4096;    // shared count array per CTA (16 KB)

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
__device__ __forceinline__ void st_vec(float* p, const float (&r)[V]) {
    if constexpr (V == 4) {
        *reinterpret_cast<float4*>(p) = make_float4(r[0], r[1], r[2], r[3]);
    } else {
        p[0] = r[0];
    }
}

template <int V>
__global__ void __launch_bounds__(OC_THREADS)
occlusion_expand_kernel(const float* __restrict__ p, int64_t ldp, const float* __restrict__ bias,
                        const float* __restrict__ w1t, int64_t ld_w1t, int n_table_rows,
                        const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                        const int32_t* __restrict__ tags, const int32_t* __restrict__ node_off,
                        const int32_t* __restrict__ v_graph, const int32_t* __restrict__ v_tag,
                        const int32_t* __restrict__ v_node_off, int width, int mode, const float* __restrict__ eps,
                        float* __restrict__ z, int64_t ldz) {
    __shared__ int cnt[OC_MAX_NODES];
    const int v = blockIdx.x;
    const int g = __ldg(v_graph + v);
    const int d = __ldg(v_tag + v);
    const int r0 = __ldg(node_off + g);
    const int n = __ldg(node_off + g + 1) - r0;
    if (n > OC_MAX_NODES) return;                         // the host rejects such batches (GNM_ERR_TOO_LARGE)
    const bool occluded = d >= 0 && d < n_table_rows;
    const float self_w = eps != nullptr ? 1.f + __ldg(eps) : 0.f;
    if (occluded) {
        for (int i = threadIdx.x; i < n; i += OC_THREADS) cnt[i] = 0;
        __syncthreads();
        // the CSR rows of the nodes tagged d list exactly the rows m with a non-zero count (the adjacency is
        // symmetric): each warp scans 32 nodes at a time and walks the row of every node it finds tagged d
        const int lane = threadIdx.x & 31;
        for (int base = (threadIdx.x >> 5) * 32; base < n; base += OC_THREADS) {
            unsigned hit = __ballot_sync(GNM_FULL_MASK, base + lane < n && __ldg(tags + r0 + base + lane) == d);
            while (hit != 0u) {
                const int r = r0 + base + __ffs(hit) - 1;
                hit &= hit - 1u;
                const int e1 = __ldg(rowptr + r + 1);
                for (int e = __ldg(rowptr + r) + lane; e < e1; e += 32) {
                    const int m = __ldg(colidx + e) - r0;
                    if (m >= 0 && m < n) atomicAdd(&cnt[m], 1);
                }
            }
        }
        __syncthreads();
    }
    const int n_vec = (width + V - 1) / V;
    const int64_t vr0 = __ldg(v_node_off + v);
    float w[V];
    for (int it = threadIdx.x; it < n * n_vec; it += OC_THREADS) {
        const int i = it / n_vec;
        const int col = (it - i * n_vec) * V;
        const int64_t r = r0 + i;
        float x[V], b[V];
        ld_vec<V>(p + r * ldp + col, x);
        if (bias != nullptr) ld_vec<V>(bias + col, b);
#pragma unroll
        for (int k = 0; k < V; ++k) x[k] = bias != nullptr ? x[k] + b[k] : x[k];
        if (occluded) {
            // c_d[m] = s_m * count + (learn_eps ? (1 + eps) [tag[m] = d] : 0); s_m formed only for a non-zero count
            const int c = cnt[i];
            float coef = 0.f;
            if (c != 0) coef = mode == 1 ? (float)c / (float)(__ldg(rowptr + r + 1) - __ldg(rowptr + r)) : (float)c;
            if (eps != nullptr && __ldg(tags + r) == d) coef += self_w;
            if (coef != 0.f) {
                ld_vec<V>(w1t + (int64_t)d * ld_w1t + col, w);
#pragma unroll
                for (int k = 0; k < V; ++k) x[k] = fmaf(-coef, w[k], x[k]);
            }
        }
        st_vec<V>(z + (vr0 + i) * ldz + col, x);
    }
}

}  // namespace

extern "C" int gnm_occlusion_expand(const float* p, int64_t ldp, const float* bias, const float* w1t, int64_t ld_w1t,
                                    int n_table_rows, const int32_t* rowptr, const int32_t* colidx, const int32_t* tags,
                                    const int32_t* node_off, int n_graphs, int n_max, const int32_t* v_graph,
                                    const int32_t* v_tag, const int32_t* v_node_off, int n_virtual, int width, int mode,
                                    const float* eps, float* z, int64_t ldz, gnm_stream_t stream) {
    if (n_table_rows < 0 || n_graphs < 0 || n_max < 0 || n_virtual < 0 || width < 0 || (mode != 0 && mode != 1))
        return GNM_ERR_BAD_ARG;
    if (n_virtual == 0 || width == 0 || n_max == 0) return GNM_OK;
    if (n_graphs == 0 || !p || !rowptr || !colidx || !tags || !node_off || !v_graph || !v_tag || !v_node_off || !z ||
        ldp < width || ldz < width || (n_table_rows > 0 && (!w1t || ld_w1t < width)))
        return GNM_ERR_BAD_ARG;
    if (n_max > OC_MAX_NODES) return GNM_ERR_TOO_LARGE;
    const bool vec4 = width % 4 == 0 && ldp % 4 == 0 && ldz % 4 == 0 && gnm_aligned16(p) && gnm_aligned16(z) &&
                      (bias == nullptr || gnm_aligned16(bias)) &&
                      (n_table_rows == 0 || (ld_w1t % 4 == 0 && gnm_aligned16(w1t)));
    cudaStream_t st = gnm_cast_stream(stream);
    gnm_count_launch(GNM_K_OCCLUSION_EXPAND);
    if (vec4)
        occlusion_expand_kernel<4><<<n_virtual, OC_THREADS, 0, st>>>(p, ldp, bias, w1t, ld_w1t, n_table_rows, rowptr,
                                                                     colidx, tags, node_off, v_graph, v_tag, v_node_off,
                                                                     width, mode, eps, z, ldz);
    else
        occlusion_expand_kernel<1><<<n_virtual, OC_THREADS, 0, st>>>(p, ldp, bias, w1t, ld_w1t, n_table_rows, rowptr,
                                                                     colidx, tags, node_off, v_graph, v_tag, v_node_off,
                                                                     width, mode, eps, z, ldz);
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}
