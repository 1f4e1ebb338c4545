// Dense-block neighbour aggregation on the tensor cores.
//
// Reference: models/graphcnn.py:154-161 / :178-182 - pooled = spmm(Adj_block, h) (+ (1+eps) h).
// Adj_block is block-diagonal with one N x N block per graph, and thresholded FC graphs are
// ~30 % dense, so gathering neighbour rows moves nnz * F * 4 bytes through L2/SMEM per layer
// (12.5 GB at B=1024, N=400, F=64) - 30x the compulsory HBM traffic. Here every block is instead
// multiplied as a dense 0/1 matrix:
//
//   P_g [N x F]  =  A_g [N x N]  .  H_g [N x F]
//
//  * A_g comes from a per-graph BITMAP (N x ceil(N/32) words, 20 KB at N=400 instead of 190 KB of
//    int32 indices); mma.sync A-fragments (bf16 0.0 / 1.0) are built in registers straight from the
//    bitmap words - the adjacency never touches shared memory.
//  * H_g is fp32; to keep fp32 results it is split on the fly into three bf16 planes
//    h = hi + mid + lo (8+8+8 significand bits: exact for normal fp32 values) that are staged in
//    shared memory ([k][feature], 144-byte pitch: conflict-free for ldmatrix) and multiplied in
//    three passes accumulating into the same fp32 accumulators. 0/1 x bf16 products are exact, so
//    the only rounding is the fp32 accumulation, as in the reference's own summation.
//  * One persistent CTA (16 warps = 4 along rows x 4 along features) per SM walks work items
//    (graph, 448-row block, 64-feature slab); K is streamed in 128-row chunks, double buffered:
//    the global loads of chunk c+1 are in flight while chunk c is in the MMA loop.
//
// Requires duplicate-free adjacency (a bitmap cannot count multiplicity); the host falls back to
// the CSR kernel otherwise. sm_100a: legacy mma.sync path (HMMA); a tcgen05 version is future work.
#include <cuda_bf16.h>

#include "gnm_common.cuh"

namespace {

constexpr int AD_KC = 128;                 // K rows per shared-memory chunk
constexpr int AD_PITCH = 72;               // bf16 per smem row: 64 features + 8 pad = 144 B
constexpr int AD_SLAB = 64;                // features per work item
constexpr int AD_PLANE = AD_KC * AD_PITCH;                  // bf16 elements per split plane
constexpr int AD_SMEM_BYTES = 2 * 3 * AD_PLANE * 2;         // two buffers x three planes

// Warp grid of one CTA: WM warps along rows x WN warps along the 64 features; every warp owns MT m16 tiles
// (rows) x NT = 8/WN n8 tiles (features). Rows per work item = WM * MT * 16.
template <int WM_, int WN_, int MT_>
struct AggDenseCfg {
    static constexpr int WM = WM_, WN = WN_, MT = MT_;
    static constexpr int NT = 8 / WN_;
    static constexpr int THREADS = WM_ * WN_ * 32;
    static constexpr int ROWS = WM_ * MT_ * 16;
    static constexpr int STAGE = AD_KC * 16 / THREADS;      // float4 loads per thread per chunk
    static_assert(NT >= 2 && (NT % 2) == 0, "ldmatrix.x4 covers two n-tiles");
    static_assert(AD_KC * 16 % THREADS == 0, "chunk must divide evenly over the CTA");
};

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                               uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3,
                                                  uint32_t smem_addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3)
                 : "r"(smem_addr));
}

// bits 0 and 1 of x -> packed bf16x2 {bit0 ? 1.0 : 0.0, bit1 ? 1.0 : 0.0}
__device__ __forceinline__ uint32_t bits_to_bf16x2(uint32_t x) {
    return (x & 1u) * 0x3F80u + (x & 2u) * 0x1FC00000u;
}

__device__ __forceinline__ void split3(float x, float& hi, float& mid, float& lo) {
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    hi = __bfloat162float(h);
    const float r1 = x - hi;
    const __nv_bfloat16 m = __float2bfloat16_rn(r1);
    mid = __bfloat162float(m);
    lo = r1 - mid;          // <= 8 significant bits left: exact in bf16
}

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<const uint32_t*>(&v);
}

struct AggDenseParams {
    const int64_t* bitmap_addr;   // [B] device addresses of each graph's bitmap (N rows x ceil(N/32) words)
    const int32_t* node_off;      // [B+1]
    const int32_t* rowptr;        // batch CSR row pointers (degrees for mode 1 / 2); may be null for mode 0
    const float* src;
    const int32_t* src_map;
    float* dst;
    const float* eps;
    const float* bias;
    int64_t ld_src, ld_dst;
    int n_graphs, n_feat, mode, n_rb, n_slabs;
};

template <class Cfg>
__global__ void __launch_bounds__(Cfg::THREADS, 1) aggregate_dense_kernel(const AggDenseParams p) {
    constexpr int AD_MT = Cfg::MT, AD_NT = Cfg::NT, AD_THREADS = Cfg::THREADS, AD_ROWS = Cfg::ROWS;
    constexpr int AD_WN = Cfg::WN, AD_WM = Cfg::WM, AD_STAGE = Cfg::STAGE;
    extern __shared__ __align__(16) unsigned char ad_smem[];
    __nv_bfloat16* sm = reinterpret_cast<__nv_bfloat16*>(ad_smem);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int warp_m = warp / AD_WN, warp_n = warp % AD_WN;
    const int g = lane >> 2, t = lane & 3;
    const int n_items = p.n_graphs * p.n_rb * p.n_slabs;
    const uint32_t sm_base = (uint32_t)__cvta_generic_to_shared(sm);
    // ldmatrix lane address components: matrix q = lane / 8, row r = lane % 8
    const int lq = lane >> 3, lr = lane & 7;
    const int ld_row = (lq & 1) * 8 + lr;           // k offset inside the 16-row k-step
    const int ld_col = warp_n * (AD_NT * 8) + (lq >> 1) * 8; // feature offset of the first n-tile pair

    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int slab = item % p.n_slabs;
        const int rb = (item / p.n_slabs) % p.n_rb;
        const int gi = item / (p.n_slabs * p.n_rb);
        const int n0 = p.node_off[gi];
        const int n = p.node_off[gi + 1] - n0;
        const int row0 = rb * AD_ROWS;
        if (row0 >= n) continue;                    // CTA-uniform
        const int f0 = slab * AD_SLAB;
        const int words = (n + 31) >> 5;
        const uint32_t* __restrict__ bm = reinterpret_cast<const uint32_t*>(p.bitmap_addr[gi]);
        const int n_chunks = (n + AD_KC - 1) / AD_KC;

        float acc[AD_MT][AD_NT][4];
#pragma unroll
        for (int i = 0; i < AD_MT; ++i)
#pragma unroll
            for (int j = 0; j < AD_NT; ++j)
#pragma unroll
                for (int k = 0; k < 4; ++k) acc[i][j][k] = 0.f;

        float4 stage[AD_STAGE];
        auto load_chunk = [&](int c) {
#pragma unroll
            for (int j = 0; j < AD_STAGE; ++j) {
                const int i = tid + AD_THREADS * j;
                const int row = i >> 4, c4 = i & 15;
                const int krow = c * AD_KC + row;
                const int col = f0 + c4 * 4;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (krow < n && col < p.n_feat) {
                    const int jr = n0 + krow;
                    const int64_t sr = p.src_map ? (int64_t)p.src_map[jr] : (int64_t)jr;
                    v = __ldg(reinterpret_cast<const float4*>(p.src + sr * p.ld_src + col));
                    if (p.mode == 2) {
                        const float w = 1.f / (float)(p.rowptr[jr + 1] - p.rowptr[jr]);
                        v.x *= w; v.y *= w; v.z *= w; v.w *= w;
                    }
                }
                stage[j] = v;
            }
        };
        auto store_chunk = [&](int buf) {
            __nv_bfloat16* base = sm + (size_t)buf * 3 * AD_PLANE;
#pragma unroll
            for (int j = 0; j < AD_STAGE; ++j) {
                const int i = tid + AD_THREADS * j;
                const int row = i >> 4, c4 = i & 15;
                float h[4], m[4], l[4];
                split3(stage[j].x, h[0], m[0], l[0]);
                split3(stage[j].y, h[1], m[1], l[1]);
                split3(stage[j].z, h[2], m[2], l[2]);
                split3(stage[j].w, h[3], m[3], l[3]);
                const int off = row * AD_PITCH + c4 * 4;
                *reinterpret_cast<uint2*>(base + off) = make_uint2(pack_bf16x2(h[0], h[1]), pack_bf16x2(h[2], h[3]));
                *reinterpret_cast<uint2*>(base + AD_PLANE + off) = make_uint2(pack_bf16x2(m[0], m[1]), pack_bf16x2(m[2], m[3]));
                *reinterpret_cast<uint2*>(base + 2 * AD_PLANE + off) = make_uint2(pack_bf16x2(l[0], l[1]), pack_bf16x2(l[2], l[3]));
            }
        };

        load_chunk(0);
        store_chunk(0);
        __syncthreads();
        for (int c = 0; c < n_chunks; ++c) {
            if (c + 1 < n_chunks) load_chunk(c + 1);
            const int k_rows = min(AD_KC, n - c * AD_KC);
            const int n_wsteps = (k_rows + 31) >> 5;               // 32 columns of A = one bitmap word
            const uint32_t buf_addr = sm_base + (uint32_t)((c & 1) * 3 * AD_PLANE * 2);
            for (int ws = 0; ws < n_wsteps; ++ws) {
                const int wi = (c * AD_KC >> 5) + ws;
                uint32_t w_lo[AD_MT], w_hi[AD_MT];
#pragma unroll
                for (int i = 0; i < AD_MT; ++i) {
                    const int r_lo = row0 + (warp_m + AD_WM * i) * 16 + g;
                    const int r_hi = r_lo + 8;
                    w_lo[i] = (r_lo < n) ? __ldg(bm + (size_t)r_lo * words + wi) : 0u;
                    w_hi[i] = (r_hi < n) ? __ldg(bm + (size_t)r_hi * words + wi) : 0u;
                }
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    const int ks = ws * 32 + half * 16;            // k offset inside the chunk
                    if (ks >= k_rows) break;                       // warp-uniform
                    uint32_t b[3][AD_NT][2];
#pragma unroll
                    for (int sp = 0; sp < 3; ++sp)
#pragma unroll
                        for (int np = 0; np < AD_NT / 2; ++np) {
                            const uint32_t addr = buf_addr +
                                (uint32_t)((sp * AD_PLANE + (ks + ld_row) * AD_PITCH + ld_col + np * 16) * 2);
                            ldmatrix_x4_trans(b[sp][2 * np][0], b[sp][2 * np][1], b[sp][2 * np + 1][0],
                                              b[sp][2 * np + 1][1], addr);
                        }
                    const int sh = half * 16 + 2 * t;
#pragma unroll
                    for (int i = 0; i < AD_MT; ++i) {
                        if (row0 + (warp_m + AD_WM * i) * 16 >= n) break;   // warp-uniform: no rows in this tile
                        const uint32_t a0 = bits_to_bf16x2(w_lo[i] >> sh);
                        const uint32_t a1 = bits_to_bf16x2(w_hi[i] >> sh);
                        const uint32_t a2 = bits_to_bf16x2(w_lo[i] >> (sh + 8));
                        const uint32_t a3 = bits_to_bf16x2(w_hi[i] >> (sh + 8));
#pragma unroll
                        for (int sp = 0; sp < 3; ++sp)
#pragma unroll
                            for (int nt = 0; nt < AD_NT; ++nt) mma_bf16_16816(acc[i][nt], a0, a1, a2, a3, b[sp][nt][0], b[sp][nt][1]);
                    }
                }
            }
            if (c + 1 < n_chunks) store_chunk((c + 1) & 1);
            __syncthreads();
        }

        // epilogue: average / eps self term / bias, fp32 float2 stores (one 32 B sector per quad)
        const float self_c = p.eps ? 1.f + __ldg(p.eps) : 0.f;
#pragma unroll
        for (int i = 0; i < AD_MT; ++i) {
            const int rbase = row0 + (warp_m + AD_WM * i) * 16;
            if (rbase >= n) break;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
                const int r = rbase + g + hh * 8;
                if (r >= n) continue;
                const int gr = n0 + r;
                float inv = 1.f;
                bool avg = false;
                if (p.mode == 1) { avg = true; inv = (float)(p.rowptr[gr + 1] - p.rowptr[gr]); }
                const int64_t sr = p.src_map ? (int64_t)p.src_map[gr] : (int64_t)gr;
#pragma unroll
                for (int nt = 0; nt < AD_NT; ++nt) {
                    const int col = f0 + warp_n * (AD_NT * 8) + nt * 8 + 2 * t;
                    if (col >= p.n_feat) continue;
                    float v0 = acc[i][nt][hh * 2], v1 = acc[i][nt][hh * 2 + 1];
                    if (avg) { v0 /= inv; v1 /= inv; }
                    if (p.eps) {
                        const float2 s = __ldg(reinterpret_cast<const float2*>(p.src + sr * p.ld_src + col));
                        v0 = fmaf(self_c, s.x, v0);
                        v1 = fmaf(self_c, s.y, v1);
                    }
                    if (p.bias) { v0 += __ldg(p.bias + col); v1 += __ldg(p.bias + col + 1); }
                    *reinterpret_cast<float2*>(p.dst + (int64_t)gr * p.ld_dst + col) = make_float2(v0, v1);
                }
            }
        }
    }
}

// One warp per row: set the bits of a graph's bitmap from its (local-column) CSR row.
__global__ void __launch_bounds__(256)
bitmap_build_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ colidx,
                    const int32_t* __restrict__ node_off, const int64_t* __restrict__ bitmap_off, int n_graphs,
                    uint32_t* __restrict__ bitmap, int32_t* __restrict__ dup_flags) {
    const int gi = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n0 = node_off[gi], n = node_off[gi + 1] - n0;
    const int words = (n + 31) >> 5;
    uint32_t* bm = bitmap + bitmap_off[gi];
    bool dup = false;
    for (int r = warp; r < n; r += 8) {
        const int s = rowptr[n0 + r], e = rowptr[n0 + r + 1];
        // rows are sorted: lane w owns word w, w+32, ...; it scans the row once per owned word range
        for (int w0 = 0; w0 < words; w0 += 32) {
            const int w = w0 + lane;
            uint32_t bits = 0;
            for (int q = s; q < e; ++q) {
                const int c = colidx[q];          // same address across the warp: broadcast
                if ((c >> 5) == w) {
                    const uint32_t b = 1u << (c & 31);
                    if (bits & b) dup = true;
                    bits |= b;
                }
            }
            if (w < words) bm[(size_t)r * words + w] = bits;
        }
    }
    if (__any_sync(GNM_FULL_MASK, dup) && lane == 0) atomicOr(&dup_flags[gi], 1);
}

}  // namespace

extern "C" int gnm_bitmap_build(const int32_t* rowptr, const int32_t* colidx, const int32_t* node_off,
                                const int64_t* bitmap_off, int n_graphs, uint32_t* bitmap, int32_t* dup_flags,
                                gnm_stream_t stream) {
    if (n_graphs < 0) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0) return GNM_OK;
    if (!rowptr || !node_off || !bitmap_off || !bitmap || !dup_flags) return GNM_ERR_BAD_ARG;
    gnm_count_launch(GNM_K_OTHER);
    bitmap_build_kernel<<<n_graphs, 256, 0, gnm_cast_stream(stream)>>>(rowptr, colidx, node_off, bitmap_off, n_graphs,
                                                                       bitmap, dup_flags);
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}

// tcgen05 / TMEM implementation (gnm_aggregate_tc.cu); GNM_ERR_TOO_LARGE = does not fit, use the mma.sync kernel
int gnm_launch_aggregate_tc(const int64_t* bitmap_addr, const int32_t* node_off, const int32_t* rowptr, int n_graphs,
                            int n_max, const float* src, int64_t ld_src, const int32_t* src_map, float* dst,
                            int64_t ld_dst, int n_feat, int mode, const float* eps, const float* bias,
                            const float* aff_coef, const float* aff_z, int64_t ld_aff_z, const GnmReluBnBwdFuse* fuse,
                            int b_shared, double* out_stats, const gnm_bn_tail* tail, const float* bn_scale,
                            const float* bn_shift, float* pooled, int64_t ld_pooled, const float* pool_scale,
                            cudaStream_t stream);

extern "C" int gnm_aggregate_dense(const int64_t* bitmap_addr, const int32_t* node_off, const int32_t* rowptr,
                                   int n_graphs, int n_max, const float* src, int64_t ld_src, const int32_t* src_map,
                                   float* dst, int64_t ld_dst, int n_feat, int mode, const float* eps,
                                   const float* bias, int impl, const float* bn_scale, const float* bn_shift,
                                   float* pooled, int64_t ld_pooled, const float* pool_scale, gnm_stream_t stream) {
    if (n_graphs < 0 || n_max < 0 || n_feat < 0 || mode < 0 || mode > 2) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || n_max == 0 || n_feat == 0) return GNM_OK;
    if (!bitmap_addr || !node_off || !src || !dst || (mode != 0 && !rowptr)) return GNM_ERR_BAD_ARG;
    if ((n_feat % 4) || (ld_src % 4) || (ld_dst % 2) || !gnm_aligned16(src) || !gnm_aligned16(dst) ||
        (bias && !gnm_aligned16(bias)))
        return GNM_ERR_ALIGN;
    if (impl < 0 || impl > 2) return GNM_ERR_BAD_ARG;
    if (bn_scale != nullptr || bn_shift != nullptr || pooled != nullptr) {
        // BatchNorm + ReLU on load (and pooling): the tcgen05 kernel only, nothing launched when it declines
        if (bn_scale == nullptr || bn_shift == nullptr) return GNM_ERR_BAD_ARG;
        if (impl == 1) return GNM_ERR_TOO_LARGE;
        if ((ld_dst % 4) || (pooled != nullptr && ((ld_pooled % 4) || !gnm_aligned16(pooled)))) return GNM_ERR_ALIGN;
        return gnm_launch_aggregate_tc(bitmap_addr, node_off, rowptr, n_graphs, n_max, src, ld_src, src_map, dst, ld_dst,
                                       n_feat, mode, eps, bias, nullptr, nullptr, 0, nullptr, 0, nullptr, nullptr, bn_scale,
                                       bn_shift, pooled, ld_pooled, pool_scale, gnm_cast_stream(stream));
    }
    if (impl != 1) {
        const int rc = gnm_launch_aggregate_tc(bitmap_addr, node_off, rowptr, n_graphs, n_max, src, ld_src, src_map, dst,
                                               ld_dst, n_feat, mode, eps, bias, nullptr, nullptr, 0, nullptr, 0, nullptr,
                                               nullptr, nullptr, nullptr, nullptr, 0, nullptr, gnm_cast_stream(stream));
        if (rc == GNM_OK || impl == 2 || (rc != GNM_ERR_TOO_LARGE && rc != GNM_ERR_ALIGN)) return rc;
    }
    AggDenseParams p;
    p.bitmap_addr = bitmap_addr; p.node_off = node_off; p.rowptr = rowptr; p.src = src; p.src_map = src_map;
    p.dst = dst; p.eps = eps; p.bias = bias; p.ld_src = ld_src; p.ld_dst = ld_dst; p.n_graphs = n_graphs;
    p.n_feat = n_feat; p.mode = mode;
    using Cfg = AggDenseCfg<4, 4, 7>;      // 16 warps: 4 per scheduler; 448 rows x 64 features per work item
    p.n_rb = (n_max + Cfg::ROWS - 1) / Cfg::ROWS;
    p.n_slabs = (n_feat + AD_SLAB - 1) / AD_SLAB;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaError_t e = cudaFuncSetAttribute(aggregate_dense_kernel<Cfg>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         AD_SMEM_BYTES);
    if (e != cudaSuccess) return (int)e;
    const int64_t items = (int64_t)n_graphs * p.n_rb * p.n_slabs;
    const int grid = (int)(items < sms ? items : sms);
    gnm_count_launch(GNM_K_AGG_MMA_SYNC);
    aggregate_dense_kernel<Cfg><<<grid, Cfg::THREADS, AD_SMEM_BYTES, gnm_cast_stream(stream)>>>(p);
    GNM_RETURN_IF_LAUNCH_FAILED();
    return GNM_OK;
}

/* Aggregation of a BatchNorm-backward result that is never materialised: dst = Agg(cA*dy + cB*z + cC) with the
 * per-channel coefficients of gnm_bn_bwd_coeffs applied to the rows as they are loaded (tcgen05 kernel only:
 * GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN when the batch does not fit it - apply gnm_bn_bwd_apply and aggregate then).
 * No (1 + eps) self term: the epilogue would add the raw dy row, not the transformed one. */
extern "C" int gnm_aggregate_dense_affine(const int64_t* bitmap_addr, const int32_t* node_off, const int32_t* rowptr,
                                          int n_graphs, int n_max, const float* dy, int64_t ld_dy, const float* z,
                                          int64_t ld_z, const float* coef, float* dst, int64_t ld_dst, int n_feat,
                                          int mode, gnm_stream_t stream) {
    if (n_graphs < 0 || n_max < 0 || n_feat < 0 || mode < 0 || mode > 2) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || n_max == 0 || n_feat == 0) return GNM_OK;
    if (!bitmap_addr || !node_off || !dy || !z || !coef || !dst || (mode != 0 && !rowptr)) return GNM_ERR_BAD_ARG;
    if ((n_feat % 4) || (ld_dy % 4) || (ld_dst % 4) || !gnm_aligned16(dy) || !gnm_aligned16(dst)) return GNM_ERR_ALIGN;
    return gnm_launch_aggregate_tc(bitmap_addr, node_off, rowptr, n_graphs, n_max, dy, ld_dy, nullptr, dst, ld_dst, n_feat,
                                   mode, nullptr, nullptr, coef, z, ld_z, nullptr, 0, nullptr, nullptr, nullptr, nullptr, nullptr,
                                   0, nullptr, gnm_cast_stream(stream));
}

/* Layer 0 on one-hot inputs when every graph of the batch carries the SAME injective tag sequence (util.py:106-116: one
 * tag per ROI, same ROI order for every subject): z0 = Agg(table[tags]) [+ (1+eps) table[tags]] + bias, i.e.
 * graphcnn.py:154-161 + the first Linear of mlp.py:48 with X_concat = stacked identities, plus the BatchNorm statistics
 * of z0 (out_stats, nullable, += [sum | sum of squares] per column) from the copy-out. The table rows are converted
 * to tensor-core operands once per CTA and stay resident for all its graphs. tcgen05 kernel only, n_feat <= 64,
 * mode 0 / 1: GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN otherwise, nothing launched (use gnm_aggregate_dense + gnm_col_stats).
 * tags: int32 [n_max], one graph's tag sequence; every graph must have n_max nodes. */
extern "C" int gnm_aggregate_dense_table(const int64_t* bitmap_addr, const int32_t* node_off, const int32_t* rowptr,
                                         int n_graphs, int n_max, const float* table, int64_t ld_table,
                                         const int32_t* tags, float* dst, int64_t ld_dst, int n_feat, int mode,
                                         const float* eps, const float* bias, double* out_stats, const gnm_bn_tail* tail,
                                         gnm_stream_t stream) {
    if (n_graphs < 0 || n_max < 0 || n_feat < 0 || mode < 0 || mode > 1) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || n_max == 0 || n_feat == 0) return GNM_OK;
    if (!bitmap_addr || !node_off || !table || !tags || !dst || (mode != 0 && !rowptr)) return GNM_ERR_BAD_ARG;
    if ((n_feat % 4) || (ld_table % 4) || (ld_dst % 4) || !gnm_aligned16(table) || !gnm_aligned16(dst) ||
        (bias && !gnm_aligned16(bias)))
        return GNM_ERR_ALIGN;
    return gnm_launch_aggregate_tc(bitmap_addr, node_off, rowptr, n_graphs, n_max, table, ld_table, tags, dst, ld_dst,
                                   n_feat, mode, eps, bias, nullptr, nullptr, 0, nullptr, 1, out_stats, tail, nullptr,
                                   nullptr, nullptr, 0, nullptr, gnm_cast_stream(stream));
}

/* Backward aggregation fused with its consumer: dy = relu'(bn(z)) * (Agg(src) [+ (1+eps) src] + d_pooled[g]*pool_scale[g]
 * + d_score[r]*u[g] + d_neg[r]) and stats += [sum dy, sum dy*xhat] - gnm_aggregate_dense followed by
 * gnm_relu_bn_bwd_reduce, without the round trip of the aggregated gradient through HBM (tcgen05 kernel only, n_feat <= 64:
 * GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN otherwise, nothing launched - run the two kernels then). */
extern "C" int gnm_aggregate_dense_relu_bn_bwd(const int64_t* bitmap_addr, const int32_t* node_off, const int32_t* rowptr,
                                               int n_graphs, int n_max, const float* src, int64_t ld_src, int n_feat,
                                               int mode, const float* eps, const float* z, int64_t ldz,
                                               const float* scale, const float* shift, const float* mean,
                                               const float* rstd, const float* d_pooled, int64_t ld_dpooled,
                                               const float* pool_scale, const float* d_score, const float* u, int64_t ldu,
                                               const float* d_neg, int64_t ld_dneg, int n_neg, float* dy, int64_t lddy,
                                               double* stats, const gnm_bn_tail* tail, gnm_stream_t stream) {
    if (n_graphs < 0 || n_max < 0 || n_feat < 0 || mode < 0 || mode > 2) return GNM_ERR_BAD_ARG;
    if (n_graphs == 0 || n_max == 0 || n_feat == 0) return GNM_OK;
    if (!bitmap_addr || !node_off || !src || !dy || !z || !scale || !shift || !mean || !rstd || (mode != 0 && !rowptr))
        return GNM_ERR_BAD_ARG;
    if (d_score != nullptr && u == nullptr) return GNM_ERR_BAD_ARG;
    if ((n_feat % 4) || (ld_src % 4) || (lddy % 4) || !gnm_aligned16(src) || !gnm_aligned16(dy)) return GNM_ERR_ALIGN;
    GnmReluBnBwdFuse f;
    f.z = z; f.ldz = ldz; f.scale = scale; f.shift = shift; f.mean = mean; f.rstd = rstd; f.d_pooled = d_pooled;
    f.ld_dpooled = ld_dpooled; f.pool_scale = pool_scale; f.d_score = d_score; f.u = u; f.ldu = ldu; f.d_neg = d_neg;
    f.ld_dneg = ld_dneg; f.n_neg = n_neg; f.stats = stats;
    return gnm_launch_aggregate_tc(bitmap_addr, node_off, rowptr, n_graphs, n_max, src, ld_src, nullptr, dy, lddy, n_feat,
                                   mode, eps, nullptr, nullptr, nullptr, 0, &f, 0, nullptr, tail, nullptr, nullptr, nullptr, 0,
                                   nullptr, gnm_cast_stream(stream));
}
