// DGI discriminator scoring (reference: models/discriminator.py:19-38, models/graphcnn.py:233-246)
// as a fused segmented reduction: nn.Bilinear(n_h, n_h, 1) is h^T W c + b = <h, u_g> + b with
// u_g = W c_g computed once per graph, instead of ATen's _trilinear expansion over all M rows.
#include <stdlib.h>

#include "gnm_common.cuh"

namespace {

constexpr int kMaxFeatPerLane = 32;   // n_h = L*F up to 1024

// bn (nullable): h_all holds each layer's PRE-BatchNorm output z and every value is read as h = relu(z*scale + shift),
// scale / shift of layer l at bn + l*ld_bn and bn + l*ld_bn + n_feat - gnm_bn_relu_readout's expression, so the result is
// bit-identical to reading the h it would have written
__device__ __forceinline__ float bn_relu(float z, float sc, float sh) { return fmaxf(fmaf(z, sc, sh), 0.f); }
__device__ __forceinline__ float4 bn_relu4(float4 z, float4 sc, float4 sh) {
    return make_float4(bn_relu(z.x, sc.x, sh.x), bn_relu(z.y, sc.y, sh.y), bn_relu(z.z, sc.z, sh.z), bn_relu(z.w, sc.w, sh.w));
}

__global__ void gather_nf_rows_kernel(const float* __restrict__ h_all, int64_t layer_stride, int n_layers, int n_feat,
                                      int64_t ldh, int n_rows, const float* __restrict__ bn, int64_t ld_bn,
                                      float* __restrict__ table) {
    const int nh = n_layers * n_feat;
    const int64_t total = (int64_t)n_rows * nh;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(i / nh), c = (int)(i % nh);
        const int l = c / n_feat, f = c % n_feat;
        float v = h_all[l * layer_stride + (int64_t)r * ldh + f];
        if (bn != nullptr) v = bn_relu(v, bn[l * ld_bn + f], bn[l * ld_bn + n_feat + f]);
        table[i] = v;
    }
}

// the [2][nh] table of scale | shift per (layer, feature) in shared memory, laid out like u_g
__device__ __forceinline__ void stage_bn(const float* __restrict__ bn, int64_t ld_bn, int n_layers, int n_feat, float* sbn) {
    const int nh = n_layers * n_feat;
    for (int i = threadIdx.x; i < nh; i += blockDim.x) {
        const int l = i / n_feat, f = i % n_feat;
        sbn[i] = bn[l * ld_bn + f];
        sbn[nh + i] = bn[l * ld_bn + n_feat + f];
    }
}

// One CTA (8 warps) per graph; u_g staged in shared memory. Vector path (F % 4 == 0): a group of F/4 lanes
// covers one node row with 128-bit loads, 32/(F/4) rows per warp at a time, all L layer slices of a row in
// flight together; scalar path otherwise (one warp per row).
template <int LPR>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(GNM_FULL_MASK, v, o);
    return v;
}

template <int LPR>   // lanes per row = F / 4 (power of two, <= 32); 0 = scalar path
__global__ void __launch_bounds__(256)
dgi_score_fwd_kernel(const float* __restrict__ h_all, int64_t layer_stride, int n_layers, int n_feat, int64_t ldh,
                     int n_rows, const float* __restrict__ u, const float* __restrict__ neg_table,
                     const int32_t* __restrict__ neg_idx, const int32_t* __restrict__ node_off,
                     const float* __restrict__ bias, const float* __restrict__ bn, int64_t ld_bn, float* __restrict__ out) {
    extern __shared__ __align__(16) float us[];    // [n_layers * n_feat] (+ [2][n_layers * n_feat] scale | shift with bn)
    __shared__ float s_neg;
    const int g = blockIdx.x;
    const int nh = n_layers * n_feat;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* sbn = us + nh;
    for (int i = threadIdx.x; i < nh; i += blockDim.x) us[i] = u[(int64_t)g * nh + i];
    if (bn != nullptr) stage_bn(bn, ld_bn, n_layers, n_feat, sbn);
    __syncthreads();
    const float b = bias ? __ldg(bias) : 0.f;
    if (warp == 0) {
        const float* nr = neg_table + (int64_t)neg_idx[g] * nh;
        float a = 0.f;
        for (int i = lane; i < nh; i += 32) a = fmaf(nr[i], us[i], a);
        a = warp_sum(a);
        if (lane == 0) s_neg = a + b;
    }
    __syncthreads();
    const float sn = s_neg;
    const int r0 = node_off[g], r1 = node_off[g + 1];
    if (LPR > 0) {
        constexpr int L = LPR > 0 ? LPR : 1;
        constexpr int RPW = 32 / L;                 // rows per warp per iteration
        const int sub = lane % L, grp = lane / L;
        for (int rb = r0 + warp * RPW; rb < r1; rb += 8 * RPW) {
            const int r = rb + grp;
            float a = 0.f;
            if (r < r1) {
                const float* hr = h_all + (int64_t)r * ldh + sub * 4;
                const float* ul = us + sub * 4;
#pragma unroll 5
                for (int l = 0; l < n_layers; ++l) {
                    float4 hv = ld_stream_f4(hr + l * layer_stride);
                    if (bn != nullptr)
                        hv = bn_relu4(hv, *reinterpret_cast<const float4*>(sbn + l * n_feat + sub * 4),
                                      *reinterpret_cast<const float4*>(sbn + nh + l * n_feat + sub * 4));
                    const float4 uv = *reinterpret_cast<const float4*>(ul + l * n_feat);
                    a = fmaf(hv.x, uv.x, a); a = fmaf(hv.y, uv.y, a); a = fmaf(hv.z, uv.z, a); a = fmaf(hv.w, uv.w, a);
                }
            }
            a = group_sum<L>(a);
            if (sub == 0 && r < r1) {
                out[r] = a + b;
                out[n_rows + r] = sn;
            }
        }
    } else {
        for (int r = r0 + warp; r < r1; r += 8) {
            float a = 0.f;
            for (int l = 0; l < n_layers; ++l) {
                const float* hr = h_all + l * layer_stride + (int64_t)r * ldh;
                const float* ul = us + l * n_feat;
                for (int f = lane; f < n_feat; f += 32) {
                    float hv = hr[f];
                    if (bn != nullptr) hv = bn_relu(hv, sbn[l * n_feat + f], sbn[nh + l * n_feat + f]);
                    a = fmaf(hv, ul[f], a);
                }
            }
            a = warp_sum(a);
            if (lane == 0) {
                out[r] = a + b;
                out[n_rows + r] = sn;
            }
        }
    }
}

__global__ void __launch_bounds__(256)
dgi_score_bwd_kernel(const float* __restrict__ h_all, int64_t layer_stride, int n_layers, int n_feat, int64_t ldh,
                     int n_rows, const float* __restrict__ d_out, const float* __restrict__ neg_table,
                     const int32_t* __restrict__ neg_idx, const int32_t* __restrict__ node_off,
                     const float* __restrict__ bn, int64_t ld_bn,
                     float* __restrict__ du, float* __restrict__ s2, double* __restrict__ d_bias) {
    extern __shared__ float acc_s[];   // [8][nh] per-warp partial du (+ [2][nh] scale | shift with bn)
    __shared__ float red[2][8];
    const int g = blockIdx.x;
    const int nh = n_layers * n_feat;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int r0 = node_off[g], r1 = node_off[g + 1];
    float* mine = acc_s + warp * nh;
    float* sbn = acc_s + 8 * nh;
    for (int i = lane; i < nh; i += 32) mine[i] = 0.f;
    if (bn != nullptr) {
        stage_bn(bn, ld_bn, n_layers, n_feat, sbn);
        __syncthreads();
    }
    __syncwarp();
    float sum1 = 0.f, sum2 = 0.f;
    for (int r = r0 + warp; r < r1; r += 8) {
        const float d1 = d_out[r];
        if (lane == 0) { sum1 += d1; sum2 += d_out[n_rows + r]; }
        for (int l = 0; l < n_layers; ++l) {
            const float* hr = h_all + l * layer_stride + (int64_t)r * ldh;
            float* ml = mine + l * n_feat;
            for (int f = lane; f < n_feat; f += 32) {
                float hv = hr[f];
                if (bn != nullptr) hv = bn_relu(hv, sbn[l * n_feat + f], sbn[nh + l * n_feat + f]);
                ml[f] = fmaf(d1, hv, ml[f]);
            }
        }
    }
    sum1 = warp_sum(sum1);
    sum2 = warp_sum(sum2);
    if (lane == 0) { red[0][warp] = sum1; red[1][warp] = sum2; }
    __syncthreads();
    float t1 = 0.f, t2 = 0.f;
    for (int w = 0; w < 8; ++w) { t1 += red[0][w]; t2 += red[1][w]; }
    const float* nr = neg_table + (int64_t)neg_idx[g] * nh;
    for (int i = threadIdx.x; i < nh; i += blockDim.x) {
        float a = 0.f;
        for (int w = 0; w < 8; ++w) a += acc_s[w * nh + i];
        du[(int64_t)g * nh + i] = fmaf(t2, nr[i], a);
    }
    if (threadIdx.x == 0) {
        s2[g] = t2;
        if (d_bias != nullptr) atomicAdd(d_bias, (double)t1 + (double)t2);
    }
}

// 64-wide fast path of the kernel above: register accumulators (one float4 per layer and lane), 128-bit streaming
// loads, two rows per warp instruction; shared memory only for the final 16-way merge.
template <int NL>
__global__ void __launch_bounds__(256)
dgi_score_bwd_vec_kernel(const float* __restrict__ h_all, int64_t layer_stride, int64_t ldh, int n_rows,
                         const float* __restrict__ d_out, const float* __restrict__ neg_table,
                         const int32_t* __restrict__ neg_idx, const int32_t* __restrict__ node_off,
                         const float* __restrict__ bn, int64_t ld_bn,
                         float* __restrict__ du, float* __restrict__ s2, double* __restrict__ d_bias) {
    constexpr int F = 64, NH = NL * F;
    __shared__ __align__(16) float part[8][NH];
    __shared__ __align__(16) float sbn[2 * NH];
    __shared__ float red[2][8];
    const int g = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int half = lane >> 4, c4 = lane & 15;
    const int r0 = node_off[g], r1 = node_off[g + 1];
    if (bn != nullptr) {
        stage_bn(bn, ld_bn, NL, F, sbn);
        __syncthreads();
    }
    float4 acc[NL];
#pragma unroll
    for (int l = 0; l < NL; ++l) acc[l] = make_float4(0.f, 0.f, 0.f, 0.f);
    float sum1 = 0.f, sum2 = 0.f;
    for (int r = r0 + warp * 2 + half; r < r1; r += 16) {
        const float d1 = d_out[r];
        if (c4 == 0) { sum1 += d1; sum2 += d_out[n_rows + r]; }
        const float* hr = h_all + (int64_t)r * ldh + c4 * 4;
        float4 hv[NL];
#pragma unroll
        for (int l = 0; l < NL; ++l) hv[l] = ld_stream_f4(hr + l * layer_stride);
        if (bn != nullptr) {
#pragma unroll
            for (int l = 0; l < NL; ++l)
                hv[l] = bn_relu4(hv[l], *reinterpret_cast<const float4*>(sbn + l * F + c4 * 4),
                                 *reinterpret_cast<const float4*>(sbn + NH + l * F + c4 * 4));
        }
#pragma unroll
        for (int l = 0; l < NL; ++l) {
            acc[l].x = fmaf(d1, hv[l].x, acc[l].x); acc[l].y = fmaf(d1, hv[l].y, acc[l].y);
            acc[l].z = fmaf(d1, hv[l].z, acc[l].z); acc[l].w = fmaf(d1, hv[l].w, acc[l].w);
        }
    }
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        acc[l].x += __shfl_xor_sync(GNM_FULL_MASK, acc[l].x, 16); acc[l].y += __shfl_xor_sync(GNM_FULL_MASK, acc[l].y, 16);
        acc[l].z += __shfl_xor_sync(GNM_FULL_MASK, acc[l].z, 16); acc[l].w += __shfl_xor_sync(GNM_FULL_MASK, acc[l].w, 16);
        if (half == 0) *reinterpret_cast<float4*>(&part[warp][l * F + c4 * 4]) = acc[l];
    }
    sum1 = warp_sum(sum1);
    sum2 = warp_sum(sum2);
    if (lane == 0) { red[0][warp] = sum1; red[1][warp] = sum2; }
    __syncthreads();
    float t1 = 0.f, t2 = 0.f;
    for (int w = 0; w < 8; ++w) { t1 += red[0][w]; t2 += red[1][w]; }
    const float* nr = neg_table + (int64_t)neg_idx[g] * NH;
    for (int i = threadIdx.x; i < NH; i += blockDim.x) {
        float a = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) a += part[w][i];
        du[(int64_t)g * NH + i] = fmaf(t2, nr[i], a);
    }
    if (threadIdx.x == 0) {
        s2[g] = t2;
        if (d_bias != nullptr) atomicAdd(d_bias, (double)t1 + (double)t2);
    }
}

// Training-step scorer (driver.Trainer). The BCE-with-logits gradient of a score is local - ds = grad_scale *
// (sigmoid(s) - y), y = 1 for the positives and 0 for the negatives (main.py:32-37) - so the pass that forms the scores
// also forms what the backward needs from n_f: d_score[r] of the positives, du_g, s2_g, d_bias, and the loss. One read
// of the L slices instead of two (dgi_score_fwd + dgi_score_bwd) and no BCE launch. Rows go to threads as in
// dgi_score_fwd_kernel<16> / dgi_score_bwd_vec_kernel and the arithmetic is theirs and bce_logits_kernel's, in the same
// order: the scores and d_score are bit-identical to that three-launch sequence; du and s2 agree to fp32 rounding (the
// negatives' gradient, formed once per graph here, can round differently), the loss differs in summation order.
template <int NL>
__global__ void __launch_bounds__(256)
dgi_score_train_kernel(const float* __restrict__ h_all, int64_t layer_stride, int64_t ldh, int n_rows,
                       const float* __restrict__ u, const float* __restrict__ neg_table,
                       const int32_t* __restrict__ neg_idx, const int32_t* __restrict__ node_off,
                       const float* __restrict__ bias, const float* __restrict__ bn, int64_t ld_bn, float grad_scale,
                       double loss_scale, float* __restrict__ out, float* __restrict__ d_score, float* __restrict__ du,
                       float* __restrict__ s2, double* __restrict__ d_bias, double* __restrict__ loss_acc) {
    constexpr int F = 64, NH = NL * F;
    __shared__ __align__(16) float us[NH];
    __shared__ __align__(16) float sbn[2 * NH];     // bn: scale | shift (shared memory, not 2 NL float4 registers)
    __shared__ __align__(16) float part[8][NH];
    __shared__ float red[2][8];
    __shared__ double lred[8];
    __shared__ float s_neg;
    const int g = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int half = lane >> 4, c4 = lane & 15;
    for (int i = threadIdx.x; i < NH; i += blockDim.x) us[i] = u[(int64_t)g * NH + i];
    if (bn != nullptr) stage_bn(bn, ld_bn, NL, F, sbn);
    __syncthreads();
    const float b = bias ? __ldg(bias) : 0.f;
    const float* nr = neg_table + (int64_t)neg_idx[g] * NH;
    if (warp == 0) {
        float a = 0.f;
        for (int i = lane; i < NH; i += 32) a = fmaf(nr[i], us[i], a);
        a = warp_sum(a);
        if (lane == 0) s_neg = a + b;
    }
    __syncthreads();
    const float sn = s_neg;
    const float y_neg = 0.f, y_pos = 1.f;
    const float d_neg = (1.f / (1.f + expf(-sn)) - y_neg) * grad_scale;     // every negative row of the graph
    const int r0 = node_off[g], r1 = node_off[g + 1];
    float4 acc[NL];
#pragma unroll
    for (int l = 0; l < NL; ++l) acc[l] = make_float4(0.f, 0.f, 0.f, 0.f);
    float sum1 = 0.f, sum2 = 0.f;
    double loss = 0.0;
    for (int rb = r0 + warp * 2; rb < r1; rb += 16) {
        const int r = rb + half;
        const bool row = r < r1;
        float4 hv[NL];
        float a = 0.f;
        if (row) {
            const float* hr = h_all + (int64_t)r * ldh + c4 * 4;
#pragma unroll
            for (int l = 0; l < NL; ++l) hv[l] = ld_stream_f4(hr + l * layer_stride);
            if (bn != nullptr) {
#pragma unroll
                for (int l = 0; l < NL; ++l)
                    hv[l] = bn_relu4(hv[l], *reinterpret_cast<const float4*>(sbn + l * F + c4 * 4),
                                     *reinterpret_cast<const float4*>(sbn + NH + l * F + c4 * 4));
            }
#pragma unroll
            for (int l = 0; l < NL; ++l) {
                const float4 uv = *reinterpret_cast<const float4*>(us + l * F + c4 * 4);
                a = fmaf(hv[l].x, uv.x, a); a = fmaf(hv[l].y, uv.y, a); a = fmaf(hv[l].z, uv.z, a); a = fmaf(hv[l].w, uv.w, a);
            }
        }
        a = group_sum<16>(a);
        if (row) {
            const float v = a + b;
            const float d1 = (1.f / (1.f + expf(-v)) - y_pos) * grad_scale;
#pragma unroll
            for (int l = 0; l < NL; ++l) {
                acc[l].x = fmaf(d1, hv[l].x, acc[l].x); acc[l].y = fmaf(d1, hv[l].y, acc[l].y);
                acc[l].z = fmaf(d1, hv[l].z, acc[l].z); acc[l].w = fmaf(d1, hv[l].w, acc[l].w);
            }
            if (c4 == 0) {
                out[r] = v;
                out[n_rows + r] = sn;
                d_score[r] = d1;
                sum1 += d1;
                sum2 += d_neg;
                loss += (double)(fmaxf(v, 0.f) - v * y_pos + log1pf(expf(-fabsf(v))));
            }
        }
    }
#pragma unroll
    for (int l = 0; l < NL; ++l) {
        acc[l].x += __shfl_xor_sync(GNM_FULL_MASK, acc[l].x, 16); acc[l].y += __shfl_xor_sync(GNM_FULL_MASK, acc[l].y, 16);
        acc[l].z += __shfl_xor_sync(GNM_FULL_MASK, acc[l].z, 16); acc[l].w += __shfl_xor_sync(GNM_FULL_MASK, acc[l].w, 16);
        if (half == 0) *reinterpret_cast<float4*>(&part[warp][l * F + c4 * 4]) = acc[l];
    }
    sum1 = warp_sum(sum1);
    sum2 = warp_sum(sum2);
    loss = warp_sum_d(loss);
    if (lane == 0) { red[0][warp] = sum1; red[1][warp] = sum2; lred[warp] = loss; }
    __syncthreads();
    float t1 = 0.f, t2 = 0.f;
    for (int w = 0; w < 8; ++w) { t1 += red[0][w]; t2 += red[1][w]; }
    for (int i = threadIdx.x; i < NH; i += blockDim.x) {
        float a = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) a += part[w][i];
        du[(int64_t)g * NH + i] = fmaf(t2, nr[i], a);
    }
    if (threadIdx.x == 0) {
        s2[g] = t2;
        atomicAdd(d_bias, (double)t1 + (double)t2);
        // the graph's negative rows all carry the score sn: their loss terms are one value times the row count
        double lt = (double)(r1 - r0) * (double)(fmaxf(sn, 0.f) - sn * y_neg + log1pf(expf(-fabsf(sn))));
        for (int w = 0; w < 8; ++w) lt += lred[w];
        atomicAdd(loss_acc, lt * loss_scale);
    }
}

__global__ void __launch_bounds__(256)
rowdot_score_kernel(const float* __restrict__ h, int64_t ldh, int n_rows, int n_feat, const float* __restrict__ u,
                    int64_t ldu, int rows_per_graph, const float* __restrict__ bias, const float* __restrict__ s_bias,
                    float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int r = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5);
    if (r >= n_rows) return;
    const float* hr = h + (int64_t)r * ldh;
    const float* ur = u + (int64_t)(r / rows_per_graph) * ldu;
    float a = 0.f;
    for (int f = lane; f < n_feat; f += 32) a = fmaf(hr[f], __ldg(ur + f), a);
    a = warp_sum(a);
    if (lane == 0) out[r] = a + (bias ? __ldg(bias) : 0.f) + (s_bias ? s_bias[r] : 0.f);
}

}  // namespace

extern "C" int gnm_gather_nf_rows(const float* h_all, int64_t layer_stride, int n_layers, int n_feat, int64_t ldh,
                                  int n_rows, const float* bn, int64_t ld_bn, float* table, gnm_stream_t stream) {
    if (n_layers < 0 || n_feat < 0 || n_rows < 0) return GNM_ERR_BAD_ARG;
    if (n_layers == 0 || n_feat == 0 || n_rows == 0) return GNM_OK;
    if (!h_all || !table) return GNM_ERR_BAD_ARG;
    const int64_t total = (int64_t)n_rows * n_layers * n_feat;
    int64_t blocks = (total + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    gnm_count_launch(GNM_K_OTHER);
    gather_nf_rows_kernel<<<(int)blocks, 256, 0, gnm_cast_stream(stream)>>>(h_all, layer_stride, n_layers, n_feat, ldh,
                                                                            n_rows, bn, ld_bn, table);
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}

extern "C" int gnm_dgi_score_fwd(const float* h_all, int64_t layer_stride, int n_layers, int n_feat, int64_t ldh,
                                 int n_rows, const float* u, const float* neg_table, const int32_t* neg_idx,
                                 const int32_t* node_off, int n_graphs, const float* bias, const float* bn, int64_t ld_bn,
                                 float* out, gnm_stream_t stream) {
    if (n_layers < 0 || n_feat < 0 || n_rows < 0 || n_graphs < 0) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || n_rows == 0) return GNM_OK;
    if (!h_all || !u || !neg_table || !neg_idx || !node_off || !out) return GNM_ERR_BAD_ARG;
    const size_t smem = (size_t)n_layers * n_feat * 4 * (bn != nullptr ? 3 : 1);
    if (smem > 48 * 1024) return GNM_ERR_TOO_LARGE;
    const int q = n_feat / 4;
    const bool vec = (n_feat % 4 == 0) && (q & (q - 1)) == 0 && q <= 32 && (ldh % 4 == 0) && (layer_stride % 4 == 0) &&
                     gnm_aligned16(h_all);
#define GNM_DGI_FWD(LPR)                                                                                             \
    do { gnm_count_launch(GNM_K_OTHER); \
    dgi_score_fwd_kernel<LPR><<<n_graphs, 256, smem, gnm_cast_stream(stream)>>>(h_all, layer_stride, n_layers, n_feat, \
                                                                                 ldh, n_rows, u, neg_table, neg_idx,   \
                                                                                 node_off, bias, bn, ld_bn, out); } while (0)
    if (!vec) GNM_DGI_FWD(0);
    else if (q == 1) GNM_DGI_FWD(1);
    else if (q == 2) GNM_DGI_FWD(2);
    else if (q == 4) GNM_DGI_FWD(4);
    else if (q == 8) GNM_DGI_FWD(8);
    else if (q == 16) GNM_DGI_FWD(16);
    else GNM_DGI_FWD(32);
#undef GNM_DGI_FWD
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}

extern "C" int gnm_dgi_score_bwd(const float* h_all, int64_t layer_stride, int n_layers, int n_feat, int64_t ldh,
                                 int n_rows, const float* d_out, const float* neg_table, const int32_t* neg_idx,
                                 const int32_t* node_off, int n_graphs, const float* bn, int64_t ld_bn, float* du, float* s2,
                                 double* d_bias, gnm_stream_t stream) {
    if (n_layers < 0 || n_feat < 0 || n_rows < 0 || n_graphs < 0) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || n_rows == 0) return GNM_OK;
    if (!h_all || !d_out || !neg_table || !neg_idx || !node_off || !du || !s2) return GNM_ERR_BAD_ARG;
    if (n_feat == 64 && n_layers >= 1 && n_layers <= 5 && (ldh & 3) == 0 && (layer_stride & 3) == 0 && gnm_aligned16(h_all)) {
#define GNM_DGI_BWD(NL) \
    do { gnm_count_launch(GNM_K_OTHER); \
    dgi_score_bwd_vec_kernel<NL><<<n_graphs, 256, 0, gnm_cast_stream(stream)>>>(h_all, layer_stride, ldh, n_rows, d_out, \
                                                                             neg_table, neg_idx, node_off, bn, ld_bn, du, s2, \
                                                                             d_bias); } while (0)
        switch (n_layers) {
            case 1: GNM_DGI_BWD(1); break;
            case 2: GNM_DGI_BWD(2); break;
            case 3: GNM_DGI_BWD(3); break;
            case 4: GNM_DGI_BWD(4); break;
            default: GNM_DGI_BWD(5); break;
        }
#undef GNM_DGI_BWD
        GNM_RETURN_IF_LAUNCH_FAILED();
        return GNM_OK;
    }
    const size_t smem = (size_t)(bn != nullptr ? 10 : 8) * n_layers * n_feat * 4;
    if (smem > 200 * 1024) return GNM_ERR_TOO_LARGE;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(dgi_score_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
    }
    gnm_count_launch(GNM_K_OTHER);
    dgi_score_bwd_kernel<<<n_graphs, 256, smem, gnm_cast_stream(stream)>>>(h_all, layer_stride, n_layers, n_feat, ldh,
                                                                           n_rows, d_out, neg_table, neg_idx, node_off,
                                                                           bn, ld_bn, du, s2, d_bias);
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}

extern "C" int gnm_dgi_score_train(const float* h_all, int64_t layer_stride, int n_layers, int n_feat, int64_t ldh,
                                   int n_rows, const float* u, const float* neg_table, const int32_t* neg_idx,
                                   const int32_t* node_off, int n_graphs, const float* bias, const float* bn,
                                   int64_t ld_bn, float grad_scale, double loss_scale, float* out, float* d_score, float* du, float* s2, double* d_bias,
                                   double* loss_acc, gnm_stream_t stream) {
    if (n_layers < 0 || n_feat < 0 || n_rows < 0 || n_graphs < 0) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || n_rows == 0) return GNM_OK;
    if (!h_all || !u || !neg_table || !neg_idx || !node_off || !out || !d_score || !du || !s2 || !d_bias || !loss_acc)
        return GNM_ERR_BAD_ARG;
    if (n_feat != 64 || n_layers < 1 || n_layers > 5) return GNM_ERR_TOO_LARGE;
    if ((ldh & 3) != 0 || (layer_stride & 3) != 0 || !gnm_aligned16(h_all)) return GNM_ERR_ALIGN;
#define GNM_DGI_TRAIN(NL) \
    do { gnm_count_launch(GNM_K_OTHER); \
    dgi_score_train_kernel<NL><<<n_graphs, 256, 0, gnm_cast_stream(stream)>>>(h_all, layer_stride, ldh, n_rows, u, neg_table, \
        neg_idx, node_off, bias, bn, ld_bn, grad_scale, loss_scale, out, d_score, du, s2, d_bias, loss_acc); } while (0)
    switch (n_layers) {
        case 1: GNM_DGI_TRAIN(1); break;
        case 2: GNM_DGI_TRAIN(2); break;
        case 3: GNM_DGI_TRAIN(3); break;
        case 4: GNM_DGI_TRAIN(4); break;
        default: GNM_DGI_TRAIN(5); break;
    }
#undef GNM_DGI_TRAIN
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}

extern "C" int gnm_rowdot_score(const float* h, int64_t ldh, int n_rows, int n_feat, const float* u, int64_t ldu,
                                int rows_per_graph, const float* bias, const float* s_bias, float* out,
                                gnm_stream_t stream) {
    if (n_rows < 0 || n_feat < 0 || rows_per_graph <= 0) return GNM_ERR_BAD_ARG;
    if (n_rows == 0) return GNM_OK;
    if (!h || !u || !out) return GNM_ERR_BAD_ARG;
    const int blocks = (n_rows + 7) / 8;
    gnm_count_launch(GNM_K_OTHER);
    rowdot_score_kernel<<<blocks, 256, 0, gnm_cast_stream(stream)>>>(h, ldh, n_rows, n_feat, u, ldu, rows_per_graph,
                                                                     bias, s_bias, out);
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}

// ---- misc -------------------------------------------------------------------------------------

extern "C" int gnm_abi_version(void) { return GNM_ABI_VERSION; }

/* 0 = the stream is not capturing, 1 = capturing, 2 = its capture was invalidated (by an operation that is not permitted
 * under capture); debugging aid for CUDA-graph capture of the step. */
extern "C" int gnm_stream_capture_status(gnm_stream_t stream, int* status) {
    cudaStreamCaptureStatus s = cudaStreamCaptureStatusNone;
    cudaError_t e = cudaStreamIsCapturing(gnm_cast_stream(stream), &s);
    if (status) *status = (int)s;
    if (e != cudaSuccess) { cudaGetLastError(); if (status && e == cudaErrorStreamCaptureInvalidated) *status = 2; }
    return GNM_OK;
}

// Off by default: measured on B200 at B = 1024 (whole step as one CUDA graph) it changes nothing - 3.69 ms with, 3.65 ms
// without (gpurun_out/r2_bench_pdl{1,0}.json): graph replay already hides the launch latency and the persistent kernels'
// tails are short. Kept as an opt-in (GNM_PDL=1 / gnm_set_pdl) for latency-bound small-batch use.
static int g_pdl = -1;                  // -1: not decided yet (environment GNM_PDL, default off)
int gnm_pdl_enabled() {
    if (g_pdl < 0) {
        const char* e = getenv("GNM_PDL");
        g_pdl = (e != nullptr && e[0] == '1') ? 1 : 0;
    }
    return g_pdl;
}
extern "C" int gnm_set_pdl(int enabled) {
    g_pdl = enabled ? 1 : 0;
    return GNM_OK;
}

static int64_t g_launch_counts[GNM_K_FAMILIES] = {0};
void gnm_count_launch(int family) {
    if (family >= 0 && family < GNM_K_FAMILIES) __atomic_fetch_add(&g_launch_counts[family], 1, __ATOMIC_RELAXED);
}
extern "C" int gnm_launch_counts(int64_t* out, int n) {
    if (!out || n < 0) return GNM_ERR_BAD_ARG;
    for (int i = 0; i < n; ++i) out[i] = i < GNM_K_FAMILIES ? __atomic_load_n(&g_launch_counts[i], __ATOMIC_RELAXED) : 0;
    return GNM_K_FAMILIES;
}

extern "C" const char* gnm_error_string(int code) {
    switch (code) {
        case GNM_OK: return "ok";
        case GNM_ERR_BAD_ARG: return "gnm: bad argument";
        case GNM_ERR_TOO_LARGE: return "gnm: problem too large for this kernel's shared-memory budget";
        case GNM_ERR_ALIGN: return "gnm: misaligned pointer or leading dimension";
        default: break;
    }
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    return "gnm: unknown error";
}

extern "C" int gnm_set_device(int dev) { return (int)cudaSetDevice(dev); }

extern "C" int gnm_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* smem_optin_bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    int v = 0;
    if (sm_count) { cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev); *sm_count = v; }
    if (cc_major) { cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMajor, dev); *cc_major = v; }
    if (cc_minor) { cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMinor, dev); *cc_minor = v; }
    if (smem_optin_bytes) { cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev); *smem_optin_bytes = v; }
    return GNM_OK;
}
