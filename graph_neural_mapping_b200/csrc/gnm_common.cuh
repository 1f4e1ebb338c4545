// Shared device helpers for libgnm (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "gnm.h"

#define GNM_FULL_MASK 0xffffffffu

#define GNM_RETURN_IF_LAUNCH_FAILED()                 \
    do {                                              \
        cudaError_t e__ = cudaGetLastError();         \
        if (e__ != cudaSuccess) return (int)e__;      \
    } while (0)

// kernel families counted by gnm_launch_counts (include/gnm.h); host-side, one increment per kernel enqueued
enum GnmKernelFamily {
    GNM_K_AGG_CSR = 0, GNM_K_AGG_MMA_SYNC, GNM_K_AGG_TC, GNM_K_LINEAR_FFMA, GNM_K_LINEAR_TC, GNM_K_LINEAR_BWD_FFMA,
    GNM_K_LINEAR_BWD_DX_TC, GNM_K_LINEAR_WGRAD_TC, GNM_K_LINEAR_WGRAD_FFMA, GNM_K_OTHER, GNM_K_LINEAR_BWD_ONEPASS_TC,
    GNM_K_SEGMENT_COLSUM, GNM_K_IG_EXPAND, GNM_K_IG_ACCUMULATE, GNM_K_IG_ATTRIBUTE, GNM_K_OCCLUSION_EXPAND,
    GNM_K_FAMILIES
};
void gnm_count_launch(int family);     // gnm_dgi.cu

// Programmatic dependent launch (PDL) for the persistent tcgen05 kernels: launched with the programmatic-stream-serialisation
// attribute, a kernel's CTAs may start on SMs the PREVIOUS kernel of the stream has already vacated and run their set-up
// (barrier init, tensor-memory allocation, weight planes, lookup tables) while its stragglers finish; pdl_wait() blocks
// until that previous kernel has completed and flushed - it stands in front of the first access to anything a
// predecessor may have produced. pdl_launch_dependents() at kernel start lets the NEXT kernel do the same to this one.
// Contract for ABI users (gnm_set_pdl): a kernel's weight operands must not be written by the kernel immediately in
// front of it in the stream (in a training step they are written once, by the optimiser, many kernels earlier).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
int gnm_pdl_enabled();                 // gnm_dgi.cu

template <typename P>
static inline cudaError_t gnm_launch_pdl(void (*kernel)(const P), int grid, int block, size_t smem, cudaStream_t st, const P& p) {
    if (!gnm_pdl_enabled()) {
        kernel<<<grid, block, smem, st>>>(p);
        return cudaGetLastError();
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid, 1, 1);
    cfg.blockDim = dim3(block, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, p);
}

static inline cudaStream_t gnm_cast_stream(gnm_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

__host__ __device__ static inline bool gnm_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(GNM_FULL_MASK, v, o);
    return v;
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(GNM_FULL_MASK, v, o);
    return v;
}

__device__ __forceinline__ int warp_inclusive_scan(int v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(GNM_FULL_MASK, v, o);
        if (lane >= o) v += t;
    }
    return v;
}

// Streaming (read-once) 128-bit load that does not allocate in L1.
__device__ __forceinline__ float4 ld_stream_f4(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}

// Optional fused consumer of the tcgen05 aggregation's output rows (gnm_aggregate_dense_relu_bn_bwd): the arguments of
// gnm_relu_bn_bwd_reduce other than the aggregated gradient itself.
struct GnmReluBnBwdFuse {
    const float* z; int64_t ldz;
    const float* scale; const float* shift; const float* mean; const float* rstd;
    const float* d_pooled; int64_t ld_dpooled; const float* pool_scale;
    const float* d_score; const float* u; int64_t ldu;
    const float* d_neg; int64_t ld_dneg; int n_neg;
    double* stats;
};
