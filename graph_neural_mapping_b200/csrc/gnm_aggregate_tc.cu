// Neighbour aggregation on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM).
//
// Same contract as aggregate_dense_kernel (gnm_aggregate_dense.cu): per graph P_g = A_g . H_g with A_g a dense
// 0/1 block expanded from the graph's bitmap and H_g (fp32) split exactly into three bf16 planes. The legacy
// mma.sync path tops out near 200 TFLOP/s on this part (measured: 16 warps change nothing, ~0.35 kMAC/clk/SM);
// tcgen05 runs the same bf16 MACs at 4 kMAC/clk/SM: the MMAs need a third of the kernel's cycles, the rest is the
// producers' instruction stream and the load latency in front of it (profiles/r1_aggregate_tcgen05*_ncu.txt).
//
// One persistent CTA per SM, work item = (graph, 64-feature slab), N <= 416 nodes:
//   * B operand = the three planes side by side as ONE [K x 192] MN-major matrix (no swizzle; core matrix
//     = 8 k-rows x 16 B; n-cores at SBO, k-cores at LBO), resident in shared memory for the whole graph
//     (154 KB). N = 192 per MMA reads the A tile once for all three planes and keeps shared-memory traffic
//     under the MMA time: 2(M+N)/(MN) = 0.026 B/MAC.
//   * A operand = 128-row x 64-column tiles of the adjacency, expanded from bitmap bytes through a 256-entry
//     byte -> 4 x bf16x2 table and written to TENSOR MEMORY (tcgen05.st, lane = row, 32 columns per stage, 4-stage
//     ring); the MMA takes A from TMEM ([a_tmem] form). A in shared memory was measured first: MMA operand fetch
//     (A 4 KB + B 6 KB per 96-cycle MMA = 107 B/clk of the 128 B/clk shared-memory pipe) starved the producers' stores.
//   * D = 128 lanes x 192 fp32 columns in TMEM (columns 0-383: two slots; A ring in columns 384-511): the epilogue
//     warps drain slot s (tcgen05.ld, hi+mid+lo summed in registers, staged through shared memory, coalesced
//     stores with average / eps self term / bias applied on the way) while the MMA thread fills slot s^1.
//   * warp roles: 0-3 epilogue, 4-11 producers (two independent groups of four; a stage belongs to one group),
//     12 MMA issue + TMEM alloc (highest warp id: issue priority); mbarriers: a_full/a_empty[4],
//     acc_full/acc_empty[2], b_free. tcgen05.commit releases A stages / publishes accumulators. The B planes
//     of an item are written chunk by chunk together with the A stages of its first row tile; item parameters and the
//     next item's first loads are requested one item / one row tile ahead.
//   * optional fusions on the same kernel: a per-column affine of two streams applied to the B rows on load
//     (gnm_aggregate_dense_affine), BatchNorm + ReLU of the layer below applied to the B rows on load together with
//     that layer's graph pooling (gnm_aggregate_dense with bn_scale), and a consumer of the output rows in the copy-out
//     (gnm_aggregate_dense_relu_bn_bwd).
//   * every wait is bounded: on a timeout the kernel raises an abort flag and drains instead of hanging.
#include <cuda_bf16.h>

#include "gnm_common.cuh"
#include "gnm_tc.cuh"
#include "gnm_bn_tail.cuh"

namespace {

constexpr int TC_KC = 64;                      // adjacency columns per A stage (4 MMAs of K = 16)
constexpr int TC_STAGES = 4;
constexpr int TC_A_COLS = TC_KC / 2;           // TMEM columns per A stage (two bf16 per 32-bit column)
constexpr int TC_A_TMEM0 = 384;                // first TMEM column of the A ring (after the two accumulator slots)
constexpr int TC_N = 192;                      // three 64-feature planes side by side
constexpr int TC_SLAB = 64;
constexpr int TC_MAX_NODES = 416;               // largest graph whose planes fit shared memory in ONE pass
constexpr int TC_K_PASS = 448;                  // larger graphs: passes over K ranges of this many nodes, dst accumulated
constexpr int TC_EPI_WARPS = 4, TC_PROD_WARPS = 8;       // 4: one epilogue group drains both slots; 8: one group per slot
constexpr int TC_PITCH = TC_SLAB + 4;                    // floats per staged output row (272 B: conflict-optimal)
constexpr int TC_STG = 32 * TC_PITCH * 4;                // bytes of one epilogue warp's staging tile
constexpr int TC_THREADS = (TC_EPI_WARPS + 1 + TC_PROD_WARPS) * 32;   // 416
constexpr int TC_MMA_WARP = TC_EPI_WARPS + TC_PROD_WARPS;              // 12
constexpr int TC_TMEM_COLS = 512;

struct AggTcParams {
    const int64_t* bitmap_addr;
    const int32_t* node_off;
    const int32_t* rowptr;
    const float* src;
    const int32_t* src_map;
    float* dst;
    const float* eps;
    const float* bias;
    int64_t ld_src, ld_dst;
    int n_graphs, n_feat, mode, n_slabs, kcores_max;
    // optional per-column affine of two streams applied to the rows on load: h = cA*src + cB*aff_z + cC (BatchNorm
    // backward folded into the aggregation of its result; aff_coef = [cA | cB | cC], each n_feat long)
    const float* aff_coef;
    const float* aff_z;
    int64_t ld_aff_z;
    // optional fused consumer of the aggregated rows (backward pass): dst = relu'(bn(rz)) * (Agg + d_pooled[g]*pool_scale[g]
    // + d_score[r]*u[g] + d_neg[r]) and its BatchNorm-backward reduction, i.e. gnm_relu_bn_bwd_reduce applied in the
    // copy-out instead of a separate pass over a materialised d_h (rz == NULL: plain aggregation)
    const float* rz; int64_t ld_rz;
    const float* r_scale; const float* r_shift; const float* r_mean; const float* r_rstd;
    const float* r_dpooled; int64_t ld_dpooled; const float* r_pool_scale;
    const float* r_dscore; const float* r_u; int64_t ld_u;
    const float* r_dneg; int64_t ld_dneg; int r_nneg;
    double* r_stats;
    // layer-0 row gather with one table shared by every graph (all graphs carry the same tag sequence): src_map holds
    // ONE graph's tags (indexed by the node's position in its graph), the B planes are converted once per CTA and
    // stay resident; out_stats (nullable) += [sum, sum of squares] per column of the rows written (BatchNorm statistics)
    int b_shared;
    double* out_stats;
    // graphs of more than TC_MAX_NODES nodes (TCV_KSPLIT variants): this launch covers adjacency columns / feature rows
    // [k_lo, k_lo + k_pass) of every graph; accumulate != 0 adds the result to what dst already holds
    int k_lo, k_pass, accumulate;
    BnTailDev tail;              // BatchNorm tail on out_stats (forward) or r_stats (fused backward); kind 0: none
    // TCV_BN: the source rows are the pre-BatchNorm output z of the layer below; h = relu(z*bn_scale + bn_shift) is
    // formed when a chunk is converted into the B planes, and pooled (nullable) receives the graph's column sums of h
    // (times pool_scale[g], nullable) - the readout of the layer below, from the rows the producers load anyway
    const float* bn_scale; const float* bn_shift;
    float* pooled; int64_t ld_pooled; const float* pool_scale;
    long long* dbg;              // nullable: per-CTA wait/busy cycle counters (profiling aid)
};

// VAR: which optional paths this instantiation carries (the others are compiled out: the three roles run different code
// at the same time, and the all-in-one kernel - 81 KB of SASS - lost 20 % to instruction fetch and dead branches):
//   TCV_FUSE relu / BatchNorm-backward consumer in the copy-out, TCV_AFF affine of two streams on the B rows,
//   TCV_MAP row map / bias / shared table / output statistics (layer 0), TCV_EPS (1 + eps) self term, TCV_AVG degree weights,
//   TCV_BN BatchNorm + ReLU of the source on load and graph pooling of the activated rows (sum pooling, one slab, alone).
enum { TCV_FUSE = 1, TCV_AFF = 2, TCV_MAP = 4, TCV_EPS = 8, TCV_AVG = 16, TCV_ALL = 31, TCV_KSPLIT = 32, TCV_BN = 64 };

// bulk prefetch of [ptr, ptr + bytes) into L2 (no destination, no completion tracking); 16-byte granularity
__device__ __forceinline__ void l2_prefetch(const void* ptr, int64_t bytes) {
    const uint32_t n = (uint32_t)(bytes & ~(int64_t)15);
    if (n == 0 || (reinterpret_cast<uintptr_t>(ptr) & 15)) return;
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(ptr), "r"(n) : "memory");
}

template <bool DBG, int VAR>
__global__ void __launch_bounds__(TC_THREADS, 1) aggregate_tc_kernel(const AggTcParams p) {
    constexpr bool kFuse = (VAR & TCV_FUSE) != 0, kAff = (VAR & TCV_AFF) != 0, kMap = (VAR & TCV_MAP) != 0,
                   kEps = (VAR & TCV_EPS) != 0, kAvg = (VAR & TCV_AVG) != 0, kSplit = (VAR & TCV_KSPLIT) != 0,
                   kBn = (VAR & TCV_BN) != 0;
    const int k_lo = kSplit ? p.k_lo : 0;
    extern __shared__ __align__(1024) unsigned char tc_smem[];
    __shared__ __align__(8) uint64_t bars[2 * TC_STAGES + 10];
    __shared__ uint32_t s_tmem;
    __shared__ int s_abort;
    uint64_t* a_full = bars;
    uint64_t* a_empty = bars + TC_STAGES;
    uint64_t* acc_full = bars + 2 * TC_STAGES;
    uint64_t* acc_empty = acc_full + 2;
    uint64_t* b_full = acc_empty + 2;
    uint64_t* b_free = b_full + 1;
    uint64_t* pool_full = b_free + 1;     // [2] TCV_BN pooling: the producers' partial column sums of an item are in place
    uint64_t* pool_empty = pool_full + 2; // [2] ... and have been read (partials double-buffered by item parity)
    const int b_ncore_stride = p.kcores_max * 128 + 16;            // SBO of B (padded: conflict-free plane fill)
    unsigned char* sm_b = tc_smem;                                  // 24 n-cores x b_ncore_stride
    float* sm_stg = reinterpret_cast<float*>(tc_smem + (size_t)24 * b_ncore_stride);   // TC_EPI_WARPS staging tiles
    // nibble -> four bf16 0/1 values (two 32-bit TMEM columns): the adjacency expansion is a table lookup. The table is
    // replicated per LANE (entry e of lane l at e * 256 + l * 8 bytes): whatever nibbles the 32 rows of a warp hold,
    // lane l always reads banks 2l, 2l + 1 - two wavefronts per LDS.64, never a conflict. (A 256-entry byte table read
    // with LDS.128 took 2.7 wavefronts per ideal one: 4.8 M of the kernel's 10.5 M shared-memory wavefronts were its
    // bank conflicts, profiles/r2_aggregate_tc_lines.txt.)
    uint2* lut = reinterpret_cast<uint2*>(tc_smem + (size_t)24 * b_ncore_stride + TC_EPI_WARPS * TC_STG);
    // fused relu / BatchNorm backward only: one more tile per epilogue warp, the z rows of its slice (cp.async)
    float* sm_zst = reinterpret_cast<float*>(tc_smem + (size_t)24 * b_ncore_stride + TC_EPI_WARPS * TC_STG + 4096);
    // affine variant only: landing area of the second stream's rows (cp.async, eight 16-byte slots per producer thread)
    float4* sm_aff = reinterpret_cast<float4*>(tc_smem + (size_t)24 * b_ncore_stride + TC_EPI_WARPS * TC_STG + 4096 +
                                               ((kFuse && p.rz != nullptr) ? TC_EPI_WARPS * TC_STG : 0));
    // pooling variant only: [2 item parities][8 producer warps][64 columns] partial column sums of the activated rows
    float* sm_pool = reinterpret_cast<float*>(tc_smem + (size_t)24 * b_ncore_stride + TC_EPI_WARPS * TC_STG + 4096);
    const bool pool_on = kBn && p.pooled != nullptr;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    pdl_launch_dependents();
    for (int i = tid; i < 16 * 32; i += TC_THREADS) {
        const uint32_t e = (uint32_t)i >> 5;
        lut[i] = make_uint2(bits2_bf16x2(e), bits2_bf16x2(e >> 2));
    }
    volatile int* abort_flag = &s_abort;
    if (tid == 0) {
        s_abort = 0;
        for (int i = 0; i < TC_STAGES; ++i) { mbar_init(&a_full[i], TC_PROD_WARPS / 2); mbar_init(&a_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 4); }
        mbar_init(b_full, TC_PROD_WARPS);
        mbar_init(b_free, 1);
        for (int i = 0; i < 2; ++i) { mbar_init(&pool_full[i], TC_PROD_WARPS); mbar_init(&pool_empty[i], 2); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == TC_MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "r"(TC_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;
    const int n_items = p.n_graphs * p.n_slabs;
    pdl_wait();          // set-up done (nothing above read global memory): now wait for the kernel in front of this one

    if (warp < TC_EPI_WARPS) {
        // ================================ epilogue: TMEM -> registers -> staging tile -> global ===========
        // Two groups of four warps (group = accumulator slot) drain alternate row tiles. Each warp sums the three
        // plane accumulators of its 32 rows, stages them in shared memory and copies them out with coalesced 128-bit
        // stores (a row-per-lane store costs 32 L1 wavefronts per instruction); the eps self term and the bias are
        // added during the copy-out, where the source rows are read coalesced as well.
        uint32_t acc_it = 0, pool_it = 0;
        long long w_acc = 0, c_drain = 0, c_copy = 0;
        const long long t_role = clock64();
        const float self_c = (kEps && p.eps) ? 1.f + __ldg(p.eps) : 0.f;
        const uint32_t my_slot = warp >> 2;
        const int q = warp & 3;
        float* stg = sm_stg + warp * (32 * TC_PITCH);
        // fused relu/BatchNorm backward (single 64-wide slab only): this lane's four columns are fixed
        const bool fuse = kFuse && p.rz != nullptr;
        const bool ostats = kMap && p.out_stats != nullptr;
        float4 r_sc = make_float4(0.f, 0.f, 0.f, 0.f), r_sh = r_sc, r_mu = r_sc, r_rs = r_sc;
        float rs1[4] = {0.f, 0.f, 0.f, 0.f}, rs2[4] = {0.f, 0.f, 0.f, 0.f};
        if (fuse && (lane & 15) * 4 < p.n_feat) {
            const int c = (lane & 15) * 4;
            r_sc = __ldg(reinterpret_cast<const float4*>(p.r_scale + c));
            r_sh = __ldg(reinterpret_cast<const float4*>(p.r_shift + c));
            r_mu = __ldg(reinterpret_cast<const float4*>(p.r_mean + c));
            r_rs = __ldg(reinterpret_cast<const float4*>(p.r_rstd + c));
        }
        for (int item = blockIdx.x; item < n_items && !*abort_flag; item += gridDim.x) {
            const int gi = item / p.n_slabs, slab = item % p.n_slabs;
            const int n0 = p.node_off[gi], n = p.node_off[gi + 1] - n0;
            const int f0 = slab * TC_SLAB;
            const int n_mt = (n + 127) >> 7;
            // K-split pass without columns for this graph: the MMA thread publishes an untouched accumulator; keep the
            // barrier protocol going but neither read it nor write dst
            const bool have_k = !kSplit || n > k_lo;
            float4 r_gp = make_float4(0.f, 0.f, 0.f, 0.f), r_uu = r_gp;
            if (fuse && (lane & 15) * 4 < p.n_feat) {
                const int c = (lane & 15) * 4;
                if (p.r_dpooled != nullptr) {
                    const float ps = p.r_pool_scale ? __ldg(p.r_pool_scale + gi) : 1.f;
                    const float4 t = __ldg(reinterpret_cast<const float4*>(p.r_dpooled + (int64_t)gi * p.ld_dpooled + c));
                    r_gp = make_float4(t.x * ps, t.y * ps, t.z * ps, t.w * ps);
                }
                if (p.r_dscore != nullptr) r_uu = __ldg(reinterpret_cast<const float4*>(p.r_u + (int64_t)gi * p.ld_u + c));
            }
            for (int mt = 0; mt < n_mt; ++mt, ++acc_it) {
                const uint32_t slot = acc_it & 1, ph = (acc_it >> 1) & 1;
                if (TC_EPI_WARPS == 8 && slot != my_slot) continue;
                float ds_row = 0.f;
                // DGI gradient of the shuffled rows (the first r_nneg rows of the batch, main.py's n_f[idx]): tiles holding
                // such rows - a handful per launch, but all of them in the first CTAs' first graphs, where a synchronous
                // load per row made those CTAs the critical path (+35 us per launch) - fetch them asynchronously into the
                // output staging tile, and the drain below adds the accumulator on top
                const bool neg_tile = fuse && p.r_dneg != nullptr && mt * 128 + q * 32 < n && n0 + mt * 128 + q * 32 < p.r_nneg;
                if (fuse && mt * 128 + q * 32 < n) {
                    // the rows this warp will mask with arrive while it waits for the accumulator: z through cp.async
                    // into its second staging tile (two rows per instruction, coalesced), d_score one row per lane
                    const int zr0 = mt * 128 + q * 32;
                    float* zst = sm_zst + warp * (32 * TC_PITCH);
                    const uint32_t zst_u32 = smem_u32(zst);
                    // lane -> (row pair member lane >> 4, float4 column lane & 15); rows advance by two per copy, addresses
                    // by a constant step (no per-row 64-bit multiply)
                    const int c4z = lane & 15;
                    const int nvz = c4z * 4 < p.n_feat ? n - zr0 - (lane >> 4) : 0;      // copy i is in range iff 2 i < nvz
                    const char* srcz = reinterpret_cast<const char*>(p.rz + (int64_t)(n0 + zr0 + (lane >> 4)) * p.ld_rz + c4z * 4);
                    const int64_t stepz = 2 * p.ld_rz * (int64_t)sizeof(float);
                    uint32_t dstz = zst_u32 + (uint32_t)(((lane >> 4) * TC_PITCH + c4z * 4) * 4);
                    if (nvz >= 31) {
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dstz), "l"(srcz) : "memory");
                            srcz += stepz;
                            dstz += 2 * TC_PITCH * 4;
                        }
                    } else {
#pragma unroll 4
                        for (int i = 0; i < 16; ++i) {
                            const bool okz = 2 * i < nvz;
                            const int nbytes = okz ? 16 : 0;
                            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dstz),
                                         "l"(okz ? srcz : reinterpret_cast<const char*>(p.rz)), "r"(nbytes) : "memory");
                            srcz += stepz;
                            dstz += 2 * TC_PITCH * 4;
                        }
                    }
                    if (neg_tile) {
                        uint32_t dstn = smem_u32(stg) + (uint32_t)(((lane >> 4) * TC_PITCH + c4z * 4) * 4);
#pragma unroll 4
                        for (int i = 0; i < 16; ++i) {
                            const int64_t gr_n = (int64_t)n0 + zr0 + 2 * i + (lane >> 4);
                            const bool okn = 2 * i < nvz && gr_n < p.r_nneg;
                            const int nbytes = okn ? 16 : 0;
                            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dstn),
                                         "l"(p.r_dneg + (okn ? gr_n * p.ld_dneg + c4z * 4 : 0)), "r"(nbytes) : "memory");
                            dstn += 2 * TC_PITCH * 4;
                        }
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");
                    if (p.r_dscore != nullptr && zr0 + lane < n) ds_row = __ldg(p.r_dscore + n0 + zr0 + lane);
                }
                if (!mbar_wait<32>(&acc_full[slot], ph, abort_flag, DBG ? &w_acc : nullptr)) break;
                tc_fence_after();
                const long long t_d0 = DBG ? clock64() : 0;
                const int row0 = mt * 128 + q * 32;              // first row (within the graph) of this warp's slice
                const int r = row0 + lane;
                const int gr = n0 + (r < n ? r : 0);
                float deg = 1.f;
                if (kAvg && p.mode == 1) deg = (float)(p.rowptr[gr + 1] - p.rowptr[gr]);
                // a warp whose 32 rows all lie beyond the graph (the tail of the last row tile) has nothing to drain
                const bool any_rows = row0 < n && have_k;
                if (neg_tile) {
                    asm volatile("cp.async.wait_group 0;" ::: "memory");
                    __syncwarp();
                }
                if (any_rows) {
#pragma unroll 1
                    for (int c0 = 0; c0 < TC_SLAB; c0 += 16) {
                        uint32_t hi[16], mid[16], lo[16];
                        const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + slot * TC_N + c0;
                        tmem_ld16(taddr, hi);
                        tmem_ld16(taddr + 64, mid);
                        tmem_ld16(taddr + 128, lo);
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                        for (int j = 0; j < 16; j += 4) {
                            float v[4];
#pragma unroll
                            for (int e = 0; e < 4; ++e)
                                v[e] = (__uint_as_float(lo[j + e]) + __uint_as_float(mid[j + e])) + __uint_as_float(hi[j + e]);
                            if (kAvg && p.mode == 1) {
#pragma unroll
                                for (int e = 0; e < 4; ++e) v[e] /= deg;
                            }
                            if (kFuse && neg_tile) {
                                const float4 a = *reinterpret_cast<const float4*>(stg + lane * TC_PITCH + c0 + j);
                                v[0] += a.x; v[1] += a.y; v[2] += a.z; v[3] += a.w;
                            }
                            *reinterpret_cast<float4*>(stg + lane * TC_PITCH + c0 + j) = make_float4(v[0], v[1], v[2], v[3]);
                        }
                    }
                }
                if (fuse) asm volatile("cp.async.wait_group 0;" ::: "memory");
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&acc_empty[slot]);       // accumulator drained: the MMA may reuse the slot
                const long long t_d1 = DBG ? clock64() : 0;
                if (DBG) c_drain += t_d1 - t_d0;
                if (any_rows) {
                    const int c4 = lane & 15;
                    const int col = f0 + c4 * 4;
                    const bool col_ok = col < p.n_feat;
                    {
                        float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (kMap && p.bias && col_ok) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias + col));
                        // Rows in batches of CB: every load of a batch (staging tile, z tile, dst / self / negative rows) is
                        // issued before the first dependent instruction, so a batch pays one shared / global round trip
                        // instead of one per row; row addresses advance by constant steps (two rows per iteration).
                        constexpr int CB = 4;
                        const int rsub = lane >> 4;
                        const int nvalid = col_ok ? n - row0 - rsub : 0;          // row 2 i + rsub of the slice exists iff 2 i < nvalid
                        const int64_t g20 = (int64_t)n0 + row0 + rsub;
                        const bool acc_dst = kSplit && p.accumulate;
                        const bool self_t = kEps && p.eps != nullptr;
                        const bool self_map = kMap && p.src_map != nullptr;
                        const bool dsc_t = fuse && p.r_dscore != nullptr;
                        const float* stg_r = stg + rsub * TC_PITCH + c4 * 4;
                        const float* z_r = kFuse ? sm_zst + warp * (32 * TC_PITCH) + rsub * TC_PITCH + c4 * 4 : nullptr;
                        char* dptr = reinterpret_cast<char*>(p.dst + g20 * p.ld_dst + col);
                        const int64_t dstep = 2 * p.ld_dst * (int64_t)sizeof(float);
                        const char* sptr = reinterpret_cast<const char*>(p.src + g20 * p.ld_src + col);
                        const int64_t sstep = 2 * p.ld_src * (int64_t)sizeof(float);
#pragma unroll 1
                        for (int i0 = 0; i0 < 16; i0 += CB) {
                            float4 vv[CB], zz[CB], oo[CB], ss[CB];
                            float dsv[CB];
#pragma unroll
                            for (int j = 0; j < CB; ++j) {
                                const int i = i0 + j;
                                const bool okr = 2 * i < nvalid;
                                // d_score of row rr lives in lane rr: EVERY lane takes part in the shuffle (narrow layers
                                // leave lanes without a column, tail tiles leave lanes without a row)
                                if (kFuse) dsv[j] = dsc_t ? __shfl_sync(GNM_FULL_MASK, ds_row, 2 * i + rsub) : 0.f;
                                vv[j] = *reinterpret_cast<const float4*>(stg_r + i * (2 * TC_PITCH));
                                if (fuse) zz[j] = *reinterpret_cast<const float4*>(z_r + i * (2 * TC_PITCH));
                                if (kSplit) {
                                    oo[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                                    if (acc_dst && okr) oo[j] = *reinterpret_cast<const float4*>(dptr + j * dstep);
                                }
                                if (kEps) {
                                    ss[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                                    if (self_t && okr) {
                                        if (self_map) {
                                            const int64_t sr = (int64_t)p.src_map[p.b_shared ? row0 + 2 * i + rsub : (int)g20 + 2 * i];
                                            ss[j] = __ldg(reinterpret_cast<const float4*>(p.src + sr * p.ld_src + col));
                                        } else {
                                            ss[j] = __ldg(reinterpret_cast<const float4*>(sptr + j * sstep));
                                        }
                                    }
                                }
                            }
#pragma unroll
                            for (int j = 0; j < CB; ++j) {
                                if (2 * (i0 + j) >= nvalid) continue;
                                float4 v = vv[j];
                                if (kSplit) { v.x += oo[j].x; v.y += oo[j].y; v.z += oo[j].z; v.w += oo[j].w; }
                                if (kEps) {
                                    v.x = fmaf(self_c, ss[j].x, v.x); v.y = fmaf(self_c, ss[j].y, v.y);
                                    v.z = fmaf(self_c, ss[j].z, v.z); v.w = fmaf(self_c, ss[j].w, v.w);
                                }
                                if (kMap) { v.x += bias4.x; v.y += bias4.y; v.z += bias4.z; v.w += bias4.w; }
                                if (ostats) {
                                    rs1[0] += v.x; rs1[1] += v.y; rs1[2] += v.z; rs1[3] += v.w;
                                    rs2[0] = fmaf(v.x, v.x, rs2[0]); rs2[1] = fmaf(v.y, v.y, rs2[1]);
                                    rs2[2] = fmaf(v.z, v.z, rs2[2]); rs2[3] = fmaf(v.w, v.w, rs2[3]);
                                }
                                if (fuse) {
                                    // gnm_relu_bn_bwd_reduce on the fly: add the readout / DGI gradients of this row, mask by
                                    // the ReLU of the layer below, accumulate sum(dy) and sum(dy * (z - mean)) (the 1 / std
                                    // factor of xhat is applied once, when the sums are folded)
                                    const float4 zv = zz[j];
                                    v.x += r_gp.x; v.y += r_gp.y; v.z += r_gp.z; v.w += r_gp.w;
                                    if (dsc_t) {
                                        const float ds = dsv[j];
                                        v.x = fmaf(ds, r_uu.x, v.x); v.y = fmaf(ds, r_uu.y, v.y);
                                        v.z = fmaf(ds, r_uu.z, v.z); v.w = fmaf(ds, r_uu.w, v.w);
                                    }
                                    v.x = (fmaf(zv.x, r_sc.x, r_sh.x) > 0.f) ? v.x : 0.f;
                                    v.y = (fmaf(zv.y, r_sc.y, r_sh.y) > 0.f) ? v.y : 0.f;
                                    v.z = (fmaf(zv.z, r_sc.z, r_sh.z) > 0.f) ? v.z : 0.f;
                                    v.w = (fmaf(zv.w, r_sc.w, r_sh.w) > 0.f) ? v.w : 0.f;
                                    rs1[0] += v.x; rs1[1] += v.y; rs1[2] += v.z; rs1[3] += v.w;
                                    rs2[0] = fmaf(v.x, zv.x - r_mu.x, rs2[0]);
                                    rs2[1] = fmaf(v.y, zv.y - r_mu.y, rs2[1]);
                                    rs2[2] = fmaf(v.z, zv.z - r_mu.z, rs2[2]);
                                    rs2[3] = fmaf(v.w, zv.w - r_mu.w, rs2[3]);
                                }
                                *reinterpret_cast<float4*>(dptr + j * dstep) = v;
                            }
                            dptr += CB * dstep;
                            sptr += CB * sstep;
                        }
                    }
                    __syncwarp();
                }
                if (DBG) c_copy += clock64() - t_d1;
            }
            if (pool_on && warp < 2) {
                // graph pooling of the layer below: the eight producer warps' partial column sums of this item (complete
                // once its first row tile was converted), added in a fixed order - one lane per column, no atomics
                const uint32_t pb = pool_it & 1, pph = (pool_it >> 1) & 1;
                if (!mbar_wait<32>(&pool_full[pb], pph, abort_flag)) break;
                const int c = warp * 32 + lane;
                const float* part = sm_pool + pb * (TC_PROD_WARPS * TC_SLAB) + c;
                float t = 0.f;
#pragma unroll
                for (int w = 0; w < TC_PROD_WARPS; ++w) t += part[w * TC_SLAB];
                if (p.pool_scale != nullptr) t *= __ldg(p.pool_scale + gi);
                if (f0 + c < p.n_feat) p.pooled[(int64_t)gi * p.ld_pooled + f0 + c] = t;
                __syncwarp();
                if (lane == 0) mbar_arrive(&pool_empty[pb]);
            }
            ++pool_it;
        }
        double* const stats_out = ostats ? p.out_stats : (fuse ? p.r_stats : nullptr);
        if (stats_out != nullptr) {
            // lanes l and l ^ 16 hold the same columns: fold, park the warp's 2 x 64 partial sums in its staging tile,
            // add the epilogue warps in a fixed order, ONE fp64 atomic per column and CTA
            __syncwarp();
            if (fuse) { rs2[0] *= r_rs.x; rs2[1] *= r_rs.y; rs2[2] *= r_rs.z; rs2[3] *= r_rs.w; }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                rs1[u] += __shfl_xor_sync(GNM_FULL_MASK, rs1[u], 16);
                rs2[u] += __shfl_xor_sync(GNM_FULL_MASK, rs2[u], 16);
                if (lane < 16) {
                    stg[lane * 4 + u] = rs1[u];
                    stg[64 + lane * 4 + u] = rs2[u];
                }
            }
            asm volatile("bar.sync 1, %0;" ::"n"(TC_EPI_WARPS * 32) : "memory");
            if (tid < 128) {
                float a = 0.f;
#pragma unroll
                for (int w = 0; w < TC_EPI_WARPS; ++w) a += sm_stg[w * (32 * TC_PITCH) + tid];
                const int c = tid & 63;
                if (c < p.n_feat) atomicAdd(&stats_out[(tid >> 6) * p.n_feat + c], (double)a);
            }
        }
        if (DBG && tid == 0) {
            p.dbg[blockIdx.x * 16 + 0] = clock64() - t_role; p.dbg[blockIdx.x * 16 + 1] = w_acc;
            p.dbg[blockIdx.x * 16 + 12] = c_drain; p.dbg[blockIdx.x * 16 + 13] = c_copy;
        }
    } else if (warp == TC_MMA_WARP) {
        // ================================ MMA issue (one thread) ==========================================
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(TC_N >> 3) << 17) |
                                   ((uint32_t)(128 >> 4) << 24);   // f32 acc, bf16 x bf16, A K-major, B MN-major
            const uint64_t db_item = umma_desc(smem_u32(sm_b), 128, (uint32_t)b_ncore_stride);
            uint32_t a_it = 0, acc_it = 0, b_it = 0;
            bool ok = true;
            long long w_af = 0, w_ae = 0;
            const long long t_role = clock64();
            for (int item = blockIdx.x; item < n_items && ok; item += gridDim.x, ++b_it) {
                const int gi = item / p.n_slabs;
                const int n = p.node_off[gi + 1] - p.node_off[gi];
                const int n_mt = (n + 127) >> 7;
                const int nk = kSplit ? max(0, min(p.k_pass, n - k_lo)) : n;
                const int ksteps_total = (nk + 15) >> 4;
                const int n_kc = (ksteps_total + 3) >> 2;
                for (int mt = 0; mt < n_mt && ok; ++mt, ++acc_it) {
                    const uint32_t slot = acc_it & 1, ph = (acc_it >> 1) & 1;
                    if (!(ok = mbar_wait(&acc_empty[slot], ph ^ 1, abort_flag, DBG ? &w_ae : nullptr))) break;
                    tc_fence_after();
                    const uint32_t d_tmem = tmem + slot * TC_N;
                    for (int kc = 0; kc < n_kc; ++kc, ++a_it) {
                        const uint32_t s = a_it % TC_STAGES, aph = (a_it / TC_STAGES) & 1;
                        if (!(ok = mbar_wait(&a_full[s], aph, abort_flag, DBG ? &w_af : nullptr))) break;
                        tc_fence_after();
                        // lean issue path: the descriptor of k-step ks differs from the chunk's first one only in
                        // its start-address field (+2 k-cores = 256 B = 16 units), the A operand by 8 TMEM columns
                        const int ks_n = min(4, ksteps_total - kc * 4);
                        const uint64_t db0 = db_item + (uint64_t)(kc * 8 * 128 >> 4);
                        const uint32_t at0 = tmem + TC_A_TMEM0 + s * TC_A_COLS;
                        umma_ts(d_tmem, at0, db0, idesc, kc ? 1u : 0u);
                        if (ks_n > 1) umma_ts(d_tmem, at0 + 8, db0 + 16, idesc, 1u);
                        if (ks_n > 2) umma_ts(d_tmem, at0 + 16, db0 + 32, idesc, 1u);
                        if (ks_n > 3) umma_ts(d_tmem, at0 + 24, db0 + 48, idesc, 1u);
                        umma_commit(&a_empty[s]);          // frees the A stage when these MMAs retire
                    }
                    if (ok) umma_commit(&acc_full[slot]);  // accumulator complete -> epilogue
                }
                if (ok) umma_commit(b_free);               // all MMAs reading this graph's B planes are done
            }
            if (DBG) { p.dbg[blockIdx.x * 16 + 2] = clock64() - t_role; p.dbg[blockIdx.x * 16 + 3] = w_af; p.dbg[blockIdx.x * 16 + 4] = w_ae; }
        }
    } else {
        // ================================ producers ========================================================
        // Stage (row tile mt, k chunk kc): the 128 x 64 adjacency tile as bf16 0/1, one row per thread, written to
        // the TMEM A ring by the four warps of one group (warp % 4 selects the 32-lane quarter a warp may touch;
        // the two groups alternate stages). During the FIRST row tile of an item every producer warp also
        // converts the item's fp32 rows of the same 64 nodes into the three bf16 B planes in shared memory, so
        // the B fill is pipelined with the MMAs. Global loads run one tile (bitmap) / two chunks (features) ahead.
        const int ptid = tid - TC_EPI_WARPS * 32;                        // 0..255
        const int grp = ptid >> 7;                                       // 0: warps 8-11, 1: warps 12-15
        const int arow = (warp & 3) * 32 + lane;                         // row of the tile = TMEM lane
        uint32_t a_it = 0, b_it = 0;
        int prev_nkc = TC_STAGES;
        bool ok = true;
        long long w_pe = 0, c_st = 0, c_fence = 0, c_arr = 0, c_bconv = 0, c_bload = 0;
        (void)c_fence; (void)c_bload;
        const long long t_role = clock64();
        // Item parameters are fetched one item ahead (their dependent global loads - node offsets, bitmap address -
        // would otherwise stall every item start), and the next item's first bitmap words and first feature chunk are
        // requested during the current item's last row tile, when the B registers are idle.
        struct ItemP { int n0, n, nk, f0, n_mt, n_kc, ksteps_total, words; const uint32_t* bm; };
        auto fetch_item = [&](int item, ItemP& q) {
            if (item < n_items) {
                const int gi = item / p.n_slabs, slab = item % p.n_slabs;
                q.n0 = p.node_off[gi];
                q.n = p.node_off[gi + 1] - q.n0;
                q.f0 = slab * TC_SLAB;
                q.bm = reinterpret_cast<const uint32_t*>(p.bitmap_addr[gi]);
            } else {
                q.n0 = 0; q.n = 0; q.f0 = 0; q.bm = nullptr;
            }
        };
        auto derive_item = [&](ItemP& q) {
            q.n_mt = (q.n + 127) >> 7;
            q.nk = kSplit ? max(0, min(p.k_pass, q.n - k_lo)) : q.n;      // K extent of this pass
            q.ksteps_total = (q.nk + 15) >> 4;
            q.n_kc = (q.ksteps_total + 3) >> 2;
            q.words = (q.n + 31) >> 5;
        };
        constexpr int MAXC = (TC_MAX_NODES + TC_KC - 1) / TC_KC;      // 7 chunks of 64 columns
        constexpr int MYC = (MAXC + 1) / 2;                           // chunks one group handles per tile
        // bitmap words (two per chunk) of this thread's row for the chunks its group produces in row tile mt
        auto load_words = [&](const ItemP& q, int mt, uint32_t it0, uint32_t (&w)[MYC][2]) {
            const int r = mt * 128 + arow;
            const bool rok = mt < q.n_mt && r < q.n;
            const int wo = k_lo >> 5;                                 // first bitmap word of this pass's column range
            const uint32_t* rowbits = q.bm + (size_t)(rok ? r : 0) * q.words + wo;
            const int first = ((it0 & 1) == (uint32_t)grp) ? 0 : 1;  // first chunk of the tile owned by this group
#pragma unroll
            for (int c = 0; c < MYC; ++c) {
                const int kc = first + 2 * c;
                w[c][0] = (rok && kc < q.n_kc && wo + 2 * kc < q.words) ? __ldg(rowbits + 2 * kc) : 0u;
                w[c][1] = (rok && kc < q.n_kc && wo + 2 * kc + 1 < q.words) ? __ldg(rowbits + 2 * kc + 1) : 0u;
            }
        };
        // A stage belongs to ONE group of four warps (the groups alternate stages and run as two independent
        // pipelines): the owner expands the adjacency tile and, during the first row tile, also converts the
        // 64 feature rows of that chunk into the three B planes.
        const int gtid = ptid & 127;
        const int lb_c4 = gtid & 15, lb_kr = gtid >> 4;      // this thread's float4 column / first node of a 64-node chunk
        float4 bq[8];
        // affine variant: this thread's column never changes within a slab - its coefficients live in registers
        float4 aff_a = make_float4(0.f, 0.f, 0.f, 0.f), aff_b = aff_a, aff_c = aff_a;
        float4 bn_sc = aff_a, bn_sh = aff_a;                 // BatchNorm variant: the same, for scale / shift
        int aff_col = -1;
        // pooling variant: this thread's share of the item's column sums (its column, rows kbase + 8u of the chunks it
        // converts), folded with lane l ^ 16 and parked per warp for the epilogue (pool_full / pool_empty, by item parity)
        float4 pacc = aff_a;
        uint32_t pool_it = 0;
        auto put_pool = [&](float4 v) -> bool {
            const uint32_t pb = pool_it & 1, pph = (pool_it >> 1) & 1;
            ++pool_it;
            v.x += __shfl_xor_sync(GNM_FULL_MASK, v.x, 16); v.y += __shfl_xor_sync(GNM_FULL_MASK, v.y, 16);
            v.z += __shfl_xor_sync(GNM_FULL_MASK, v.z, 16); v.w += __shfl_xor_sync(GNM_FULL_MASK, v.w, 16);
            if (!mbar_wait<32>(&pool_empty[pb], pph ^ 1, abort_flag)) return false;
            if (lane < 16) *reinterpret_cast<float4*>(sm_pool + pb * (TC_PROD_WARPS * TC_SLAB) + (ptid >> 5) * TC_SLAB + lane * 4) = v;
            __syncwarp();
            if (lane == 0) mbar_arrive(&pool_full[pb]);
            return true;
        };
        // The second stream (aff_z) lands in shared memory through cp.async and meets the first (registers, bq) only when
        // the chunk is converted: forming cA*src + cB*z + cC right behind the loads made every chunk wait for DRAM
        // (B fill 130 k of 292 k cycles per CTA, 164 us per launch against 96 us for the plain variant).
        float4* my_aff = sm_aff + ptid;                      // slot u at my_aff[u * 256]
        const uint32_t my_aff_u32 = smem_u32(my_aff);
        const bool aff_on = kAff && p.aff_coef != nullptr;
        auto load_b = [&](const ItemP& q, int kc) {
            const int col = q.f0 + lb_c4 * 4;
            const bool ok0 = kc < q.n_kc && col < p.n_feat;
            const int kbase = kc * TC_KC + lb_kr;             // rows kbase, kbase + 8, ... of the graph
            if (kAff && ok0 && p.aff_coef != nullptr && aff_col != col) {
                aff_a = __ldg(reinterpret_cast<const float4*>(p.aff_coef + col));
                aff_b = __ldg(reinterpret_cast<const float4*>(p.aff_coef + p.n_feat + col));
                aff_c = __ldg(reinterpret_cast<const float4*>(p.aff_coef + 2 * p.n_feat + col));
                aff_col = col;
            }
            if (kBn && ok0 && aff_col != col) {
                bn_sc = __ldg(reinterpret_cast<const float4*>(p.bn_scale + col));
                bn_sh = __ldg(reinterpret_cast<const float4*>(p.bn_shift + col));
                aff_col = col;
            }
            // a chunk that was requested but never converted (a group without a chunk in a one-chunk graph) must not
            // race the new requests for the same landing slots
            if (kAff && aff_on) asm volatile("cp.async.wait_group 0;" ::: "memory");
            const float* rowp = p.src + (int64_t)(q.n0 + k_lo + kbase) * p.ld_src + col;
            const float* zrow = kAff ? p.aff_z + (int64_t)(q.n0 + k_lo + kbase) * p.ld_aff_z + col : nullptr;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int k = kbase + u * 8;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ok0 && k < q.nk) {
                    if (kMap && p.src_map) {
                        const int64_t sr = (int64_t)p.src_map[p.b_shared ? k : q.n0 + k_lo + k];
                        v = __ldg(reinterpret_cast<const float4*>(p.src + sr * p.ld_src + col));
                    } else {
                        v = __ldg(reinterpret_cast<const float4*>(rowp + (int64_t)(u * 8) * p.ld_src));
                    }
                    if (kAvg && p.mode == 2 && !aff_on) {
                        const int jr = q.n0 + k_lo + k;
                        const float w = 1.f / (float)(p.rowptr[jr + 1] - p.rowptr[jr]);
                        v.x *= w; v.y *= w; v.z *= w; v.w *= w;
                    }
                }
                if (kAff && aff_on) {
                    const bool okz = ok0 && k < q.nk;
                    const int nbytes = okz ? 16 : 0;
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(my_aff_u32 + (uint32_t)(u * 256 * 16)),
                                 "l"(okz ? zrow + (int64_t)(u * 8) * p.ld_aff_z : p.aff_z), "r"(nbytes) : "memory");
                }
                bq[u] = v;
            }
            if (kAff && aff_on) asm volatile("cp.async.commit_group;" ::: "memory");
        };
        ItemP cur, nxt;
        fetch_item(blockIdx.x, cur);
        derive_item(cur);
        bool preloaded = false;                  // w_cur / bq already hold this item's first words / first chunk
        uint32_t w_cur[MYC][2], w_nxt[MYC][2];
        for (int item = blockIdx.x; item < n_items && ok; item += gridDim.x, ++b_it) {
            fetch_item(item + gridDim.x, nxt);   // in flight during this whole item
            const int n = cur.n, n_mt = cur.n_mt, n_kc = cur.n_kc, ksteps_total = cur.ksteps_total;
            // shared table: only this CTA's first item converts (and loads) the B planes
            const bool do_b = !(kMap && p.b_shared) || item == (int)blockIdx.x;
            if (!preloaded) {
                load_words(cur, 0, a_it, w_cur);
                if (do_b) load_b(cur, ((a_it & 1) == (uint32_t)grp) ? 0 : 1);
            }
            preloaded = false;
            bool first_b = true;
            for (int mt = 0; mt < n_mt && ok; ++mt) {
                const long long tt0 = DBG ? clock64() : 0;
                if (ptid == 0 && mt == (n_mt > 1 ? 1 : 0) && item + (int)gridDim.x < n_items) {
                    // The NEXT item's feature rows and bitmap are pulled into L2 now, two to three row tiles before its
                    // first loads: one bulk L2 prefetch per stream (the rows of a graph are contiguous), so that the
                    // register loads in front of the B conversion (only one chunk ahead - there are no registers for
                    // more) and the bitmap word loads hit L2 instead of waiting for DRAM. `nxt` was requested at the
                    // start of this item and has arrived by now.
                    if (!(kMap && p.b_shared) && !(kMap && p.src_map) && p.ld_src == p.n_feat) {
                        l2_prefetch(p.src + (int64_t)nxt.n0 * p.ld_src, (int64_t)nxt.n * p.n_feat * 4);
                        if (kAff && p.aff_z != nullptr && p.ld_aff_z == p.n_feat)
                            l2_prefetch(p.aff_z + (int64_t)nxt.n0 * p.ld_aff_z, (int64_t)nxt.n * p.n_feat * 4);
                    }
                    if (nxt.bm != nullptr) l2_prefetch(nxt.bm, (int64_t)nxt.n * ((nxt.n + 31) >> 5) * 4);
                }
                if (mt == n_mt - 1 && mt > 0 && item + (int)gridDim.x < n_items) {
                    // last row tile: the B registers are idle (conversion happens in tile 0 only)
                    derive_item(nxt);
                    const uint32_t it_next = a_it + n_kc;                 // ring position at the next item's start
                    load_words(nxt, 0, it_next, w_nxt);
                    if (!(kMap && p.b_shared)) load_b(nxt, ((it_next & 1) == (uint32_t)grp) ? 0 : 1);
                    preloaded = true;
                } else {
                    load_words(cur, mt + 1, a_it + n_kc, w_nxt);
                }
                const int first = ((a_it & 1) == (uint32_t)grp) ? 0 : 1;
                if (DBG) c_bload += clock64() - tt0;                // tile head: next tile's / next item's loads issued
                // this group's stages only (every other one; the skipped iterations of a full-range loop cost 9 % of the
                // kernel's stall samples in branch resolution)
                const uint32_t a_it0 = a_it;
                a_it += (uint32_t)n_kc;
#pragma unroll 1
                for (int kc = first; kc < n_kc; kc += 2) {
                    const uint32_t ai = a_it0 + (uint32_t)kc;
                    const uint32_t s = ai % TC_STAGES, aph = (ai / TC_STAGES) & 1;
                    const long long tw0 = DBG ? clock64() : 0;
                    if (!(ok = mbar_wait<32>(&a_empty[s], aph ^ 1, abort_flag, DBG ? &w_pe : nullptr))) break;
                    if (DBG) c_fence += clock64() - tw0;            // whole wait call, fast path included
                    if (mt == 0 && do_b) {
                        // the previous item's MMAs on these B rows retired at least TC_STAGES stages ago, unless
                        // that item had fewer k chunks than the ring: then wait for its explicit b_free commit
                        if (first_b && prev_nkc < TC_STAGES) {
                            if (!(ok = mbar_wait<32>(b_free, (b_it & 1) ^ 1, abort_flag))) break;
                        }
                        first_b = false;
                        const long long tb0 = DBG ? clock64() : 0;
                        if (kAff && aff_on) {
                            // the chunk's second stream has landed (one group per chunk and thread): h = cA*src + cB*z + cC
                            asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
                            for (int u = 0; u < 8; ++u) {
                                const int k = kc * TC_KC + lb_kr + u * 8;
                                const float4 zv = my_aff[u * 256];
                                float4 v = bq[u];
                                v.x = fmaf(aff_a.x, v.x, fmaf(aff_b.x, zv.x, aff_c.x)); v.y = fmaf(aff_a.y, v.y, fmaf(aff_b.y, zv.y, aff_c.y));
                                v.z = fmaf(aff_a.z, v.z, fmaf(aff_b.z, zv.z, aff_c.z)); v.w = fmaf(aff_a.w, v.w, fmaf(aff_b.w, zv.w, aff_c.w));
                                if (k >= cur.nk || lb_c4 * 4 + cur.f0 >= p.n_feat) v = make_float4(0.f, 0.f, 0.f, 0.f);
                                if (kAvg && p.mode == 2 && k < cur.nk) {
                                    const int jr = cur.n0 + k_lo + k;
                                    const float w = 1.f / (float)(p.rowptr[jr + 1] - p.rowptr[jr]);
                                    v.x *= w; v.y *= w; v.z *= w; v.w *= w;
                                }
                                bq[u] = v;
                            }
                        }
                        if (kBn) {
                            // h = relu(z*scale + shift) with the readout's expression: bit-identical to aggregating the
                            // materialised h. Rows past the graph and columns past n_feat were loaded as 0, and
                            // relu(0*scale + shift) is not 0: they are zeroed AFTER the affine, for the planes and the sums
                            const bool col_in = lb_c4 * 4 + cur.f0 < p.n_feat;
#pragma unroll
                            for (int u = 0; u < 8; ++u) {
                                const int k = kc * TC_KC + lb_kr + u * 8;
                                float4 v = bq[u];
                                v.x = fmaxf(fmaf(v.x, bn_sc.x, bn_sh.x), 0.f); v.y = fmaxf(fmaf(v.y, bn_sc.y, bn_sh.y), 0.f);
                                v.z = fmaxf(fmaf(v.z, bn_sc.z, bn_sh.z), 0.f); v.w = fmaxf(fmaf(v.w, bn_sc.w, bn_sh.w), 0.f);
                                if (k >= cur.nk || !col_in) v = make_float4(0.f, 0.f, 0.f, 0.f);
                                if (pool_on) { pacc.x += v.x; pacc.y += v.y; pacc.z += v.z; pacc.w += v.w; }
                                bq[u] = v;
                            }
                        }
#pragma unroll
                        for (int u = 0; u < 8; ++u) {
                            const int k = kc * TC_KC + lb_kr + u * 8, c4 = lb_c4;
                            if (k >= ksteps_total * 16) continue;
                            uint32_t h0, m0, l0, h1, m1, l1;
                            split3x2(bq[u].x, bq[u].y, h0, m0, l0);
                            split3x2(bq[u].z, bq[u].w, h1, m1, l1);
                            unsigned char* dstp = sm_b + (size_t)(c4 >> 1) * b_ncore_stride + (k >> 3) * 128 + (k & 7) * 16 + (c4 & 1) * 8;
                            *reinterpret_cast<uint2*>(dstp) = make_uint2(h0, h1);
                            *reinterpret_cast<uint2*>(dstp + 8 * (size_t)b_ncore_stride) = make_uint2(m0, m1);
                            *reinterpret_cast<uint2*>(dstp + 16 * (size_t)b_ncore_stride) = make_uint2(l0, l1);
                        }
                        if (kc + 2 < n_kc) load_b(cur, kc + 2);
                        fence_async_smem();
                        if (DBG) c_bconv += clock64() - tb0;
                    }
                    const long long tq0 = DBG ? clock64() : 0;
                    // rows beyond the graph are never read back from the accumulator, so their A rows may hold
                    // anything: a warp whose whole lane quarter is past the last node skips the expansion
                    if (mt * 128 + (warp & 3) * 32 < n) {
                        // 64 bits -> 32 registers of bf16 pairs -> 32 TMEM columns of this row
                        const uint32_t taddr = tmem + ((uint32_t)((warp & 3) * 32) << 16) + TC_A_TMEM0 + s * TC_A_COLS;
#pragma unroll
                        const uint2* my_lut = lut + lane;
                        for (int hw = 0; hw < 2; ++hw) {
                            uint32_t v[16];
                            const uint32_t w32 = w_cur[0][hw];
#pragma unroll
                            for (int b = 0; b < 8; ++b) {
                                const uint2 t2 = my_lut[((w32 >> (4 * b)) & 15u) * 32];
                                v[2 * b] = t2.x; v[2 * b + 1] = t2.y;
                            }
                            tmem_st16(taddr + hw * 16, v);
                        }
#pragma unroll
                        for (int c = 0; c + 1 < MYC; ++c) { w_cur[c][0] = w_cur[c + 1][0]; w_cur[c][1] = w_cur[c + 1][1]; }
                        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                    }
                    const long long tq1 = DBG ? clock64() : 0;
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&a_full[s]);
                    if (DBG) { const long long tq3 = clock64(); c_st += tq1 - tq0; c_arr += tq3 - tq1; }
                }
                if (pool_on && mt == 0 && ok) {
                    ok = put_pool(pacc);
                    pacc = make_float4(0.f, 0.f, 0.f, 0.f);
                }
                const long long tt1 = DBG ? clock64() : 0;
#pragma unroll
                for (int c = 0; c < MYC; ++c) { w_cur[c][0] = w_nxt[c][0]; w_cur[c][1] = w_nxt[c][1]; }
                if (DBG) c_bload += clock64() - tt1;                // tile tail: the prefetched words must have arrived
            }
            if (pool_on && n_mt == 0 && ok) ok = put_pool(make_float4(0.f, 0.f, 0.f, 0.f));     // empty graph: sums 0
            prev_nkc = n_kc;
            if (!preloaded) derive_item(nxt);
            cur = nxt;
        }
        if (DBG && ptid == 0) {
            p.dbg[blockIdx.x * 16 + 5] = clock64() - t_role; p.dbg[blockIdx.x * 16 + 6] = w_pe;
            p.dbg[blockIdx.x * 16 + 7] = c_st; p.dbg[blockIdx.x * 16 + 8] = c_fence; p.dbg[blockIdx.x * 16 + 9] = c_arr;
            p.dbg[blockIdx.x * 16 + 10] = c_bconv; p.dbg[blockIdx.x * 16 + 11] = c_bload;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == TC_MMA_WARP) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TC_TMEM_COLS) : "memory");
    }
    if (kFuse || kMap) bn_tail_run(p.tail);
}

template <bool DBG, int VAR>
cudaError_t launch_variant(const AggTcParams& p, int grid, int smem, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(aggregate_tc_kernel<DBG, VAR>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return e;
    gnm_count_launch(GNM_K_AGG_TC);
    return gnm_launch_pdl<AggTcParams>(aggregate_tc_kernel<DBG, VAR>, grid, TC_THREADS, smem, stream, p);
}

}  // namespace

static long long* g_tc_dbg_host = nullptr;   // profiling aid, see gnm_aggregate_tc_set_debug

// Returns GNM_OK after launching, or GNM_ERR_TOO_LARGE when the batch does not fit this kernel (caller falls back).
int gnm_launch_aggregate_tc(const int64_t* bitmap_addr, const int32_t* node_off, const int32_t* rowptr, int n_graphs,
                            int n_max, const float* src, int64_t ld_src, const int32_t* src_map, float* dst,
                            int64_t ld_dst, int n_feat, int mode, const float* eps, const float* bias,
                            const float* aff_coef, const float* aff_z, int64_t ld_aff_z, const GnmReluBnBwdFuse* fuse,
                            int b_shared, double* out_stats, const gnm_bn_tail* tail, const float* bn_scale,
                            const float* bn_shift, float* pooled, int64_t ld_pooled, const float* pool_scale,
                            cudaStream_t stream) {
    if (bn_scale != nullptr) {
        // BatchNorm + ReLU on load (+ pooling): single pass, sum pooling, one slab, no self term / row map / other fusion
        if (bn_shift == nullptr) return GNM_ERR_BAD_ARG;
        if (n_max > TC_MAX_NODES || n_feat > TC_SLAB || mode != 0 || eps != nullptr || src_map != nullptr || bias != nullptr ||
            fuse != nullptr || aff_coef != nullptr || b_shared || out_stats != nullptr || tail != nullptr)
            return GNM_ERR_TOO_LARGE;
        if (!gnm_aligned16(bn_scale) || !gnm_aligned16(bn_shift)) return GNM_ERR_ALIGN;
    }
    // graphs above TC_MAX_NODES nodes: K-split passes (plain / eps / row-map variants of sum pooling and of the transposed
    // average, mode 2); the fused consumers, the shared table and the forward average (division of the TOTAL) stay single-pass
    const bool ksplit = n_max > TC_MAX_NODES;
    if (ksplit && (n_max > 8192 || fuse != nullptr || aff_coef != nullptr || out_stats != nullptr || b_shared || mode == 1 ||
                   tail != nullptr))
        return GNM_ERR_TOO_LARGE;
    if (tail != nullptr && out_stats == nullptr && (fuse == nullptr || fuse->stats == nullptr)) return GNM_ERR_BAD_ARG;
    if ((out_stats != nullptr || b_shared) && (n_feat > TC_SLAB || fuse != nullptr || aff_coef != nullptr || mode == 2))
        return GNM_ERR_TOO_LARGE;              // one 64-wide slab per lane; a shared table has no per-graph row weights
    if (b_shared && src_map == nullptr) return GNM_ERR_BAD_ARG;
    if (fuse != nullptr) {
        if (n_feat > TC_SLAB) return GNM_ERR_TOO_LARGE;             // the fused reduction keeps one 64-wide slab per lane
        if ((fuse->ldz % 4) || !gnm_aligned16(fuse->z) || !gnm_aligned16(fuse->scale) || !gnm_aligned16(fuse->shift) ||
            !gnm_aligned16(fuse->mean) || !gnm_aligned16(fuse->rstd) ||
            (fuse->d_pooled && ((fuse->ld_dpooled % 4) || !gnm_aligned16(fuse->d_pooled))) ||
            (fuse->d_score && ((fuse->ldu % 4) || !gnm_aligned16(fuse->u))) ||
            (fuse->d_neg && ((fuse->ld_dneg % 4) || !gnm_aligned16(fuse->d_neg))))
            return GNM_ERR_ALIGN;
    }
    if (aff_coef != nullptr && (aff_z == nullptr || (ld_aff_z % 4) || !gnm_aligned16(aff_z) || !gnm_aligned16(aff_coef)))
        return GNM_ERR_ALIGN;
    if ((ld_dst % 4) || (ld_src % 4) || (n_feat % 4)) return GNM_ERR_ALIGN;
    int dev = 0, sms = 148, major = 0, smem_cap = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    if (major != 10) return GNM_ERR_TOO_LARGE;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cudaDeviceGetAttribute(&smem_cap, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    AggTcParams p;
    p.bitmap_addr = bitmap_addr; p.node_off = node_off; p.rowptr = rowptr; p.src = src; p.src_map = src_map;
    p.dst = dst; p.eps = eps; p.bias = bias; p.ld_src = ld_src; p.ld_dst = ld_dst; p.n_graphs = n_graphs;
    p.n_feat = n_feat; p.mode = mode;
    p.aff_coef = aff_coef; p.aff_z = aff_z; p.ld_aff_z = ld_aff_z;
    p.rz = nullptr; p.ld_rz = 0; p.r_scale = p.r_shift = p.r_mean = p.r_rstd = nullptr;
    p.r_dpooled = nullptr; p.ld_dpooled = 0; p.r_pool_scale = nullptr; p.r_dscore = nullptr; p.r_u = nullptr; p.ld_u = 0;
    p.r_dneg = nullptr; p.ld_dneg = 0; p.r_nneg = 0; p.r_stats = nullptr;
    if (fuse != nullptr) {
        p.rz = fuse->z; p.ld_rz = fuse->ldz; p.r_scale = fuse->scale; p.r_shift = fuse->shift; p.r_mean = fuse->mean;
        p.r_rstd = fuse->rstd; p.r_dpooled = fuse->d_pooled; p.ld_dpooled = fuse->ld_dpooled;
        p.r_pool_scale = fuse->pool_scale; p.r_dscore = fuse->d_score; p.r_u = fuse->u; p.ld_u = fuse->ldu;
        p.r_dneg = fuse->d_neg; p.ld_dneg = fuse->ld_dneg; p.r_nneg = fuse->n_neg; p.r_stats = fuse->stats;
    }
    p.b_shared = b_shared; p.out_stats = out_stats;
    p.k_lo = 0; p.k_pass = 0; p.accumulate = 0;
    p.bn_scale = bn_scale; p.bn_shift = bn_shift;
    p.pooled = bn_scale != nullptr ? pooled : nullptr; p.ld_pooled = ld_pooled; p.pool_scale = pool_scale;
    const int trc = bn_tail_args(tail, out_stats != nullptr ? out_stats : (fuse ? fuse->stats : nullptr), n_feat, &p.tail);
    if (trc != GNM_OK) return trc;
    p.dbg = g_tc_dbg_host;
    p.n_slabs = (n_feat + TC_SLAB - 1) / TC_SLAB;
    p.kcores_max = (((ksplit ? TC_K_PASS : n_max) + 15) / 16) * 2;
    // B planes + staging + LUT (+ the z tiles of the fused relu / BatchNorm backward)
    const int smem = 24 * (p.kcores_max * 128 + 16) + TC_EPI_WARPS * TC_STG + 4096 + 1024 + (fuse ? TC_EPI_WARPS * TC_STG : 0) +
                     (aff_coef ? TC_PROD_WARPS * 32 * 8 * 16 : 0) + (p.pooled ? 2 * TC_PROD_WARPS * TC_SLAB * 4 : 0);
    if (smem > smem_cap - 1024) return GNM_ERR_TOO_LARGE;
    const int64_t items = (int64_t)n_graphs * p.n_slabs;
    const int grid = (int)(items < sms ? items : sms);
    // the paths this call needs; the lean instantiations cover sum pooling (mode 0), everything else takes the all-in-one
    int var = (fuse ? TCV_FUSE : 0) | (aff_coef ? TCV_AFF : 0) | ((src_map || bias || out_stats || b_shared) ? TCV_MAP : 0) |
              (eps ? TCV_EPS : 0) | (mode != 0 ? TCV_AVG : 0);
    cudaError_t e;
    if (ksplit) {
        // pass 0 carries the self term and the bias, later passes add their columns' contribution to dst
        for (int k_lo = 0; k_lo < n_max; k_lo += TC_K_PASS) {
            p.k_lo = k_lo; p.k_pass = TC_K_PASS; p.accumulate = k_lo > 0;
            if (k_lo > 0) { p.eps = nullptr; p.bias = nullptr; }
            const int v2 = ((src_map || bias) ? TCV_MAP : 0) | (eps ? TCV_EPS : 0);
            if (mode == 2) e = launch_variant<false, TCV_KSPLIT | TCV_AVG | TCV_MAP | TCV_EPS>(p, grid, smem, stream);
            else if (v2 == 0) e = launch_variant<false, TCV_KSPLIT>(p, grid, smem, stream);
            else if (v2 == TCV_EPS) e = launch_variant<false, TCV_KSPLIT | TCV_EPS>(p, grid, smem, stream);
            else e = launch_variant<false, TCV_KSPLIT | TCV_MAP | TCV_EPS>(p, grid, smem, stream);
            if (e != cudaSuccess) return (int)e;
        }
        return GNM_OK;
    }
    if (bn_scale != nullptr) {
        e = p.dbg != nullptr ? launch_variant<true, TCV_BN>(p, grid, smem, stream) : launch_variant<false, TCV_BN>(p, grid, smem, stream);
        return e == cudaSuccess ? GNM_OK : (int)e;
    }
    if (p.dbg != nullptr) {
        e = var == 0 ? launch_variant<true, 0>(p, grid, smem, stream)
            : var == TCV_FUSE ? launch_variant<true, TCV_FUSE>(p, grid, smem, stream)
            : var == TCV_MAP ? launch_variant<true, TCV_MAP>(p, grid, smem, stream)
            : var == TCV_AFF ? launch_variant<true, TCV_AFF>(p, grid, smem, stream) : launch_variant<true, TCV_ALL>(p, grid, smem, stream);
        return e == cudaSuccess ? GNM_OK : (int)e;
    }
    switch (var) {
        case 0: e = launch_variant<false, 0>(p, grid, smem, stream); break;
        case TCV_EPS: e = launch_variant<false, TCV_EPS>(p, grid, smem, stream); break;
        case TCV_FUSE: e = launch_variant<false, TCV_FUSE>(p, grid, smem, stream); break;
        case TCV_FUSE | TCV_EPS: e = launch_variant<false, TCV_FUSE | TCV_EPS>(p, grid, smem, stream); break;
        case TCV_AFF: e = launch_variant<false, TCV_AFF>(p, grid, smem, stream); break;
        case TCV_MAP: e = launch_variant<false, TCV_MAP>(p, grid, smem, stream); break;
        case TCV_MAP | TCV_EPS: e = launch_variant<false, TCV_MAP | TCV_EPS>(p, grid, smem, stream); break;
        default: e = launch_variant<false, TCV_ALL>(p, grid, smem, stream); break;
    }
    return e == cudaSuccess ? GNM_OK : (int)e;
}

/* 1 if any tcgen05 aggregation launch since the last call hit a wait timeout (its output is then invalid).
 * Synchronises the device; for tests and smoke checks. */
int gnm_linear_tc_abort_flag(int* aborted);     // gnm_linear_tc.cu
int gnm_linear_bwd_tc_abort_flag(int* aborted); // gnm_linear_bwd_tc.cu

extern "C" int gnm_aggregate_tc_status(int* aborted) {
    int v = 0, zero = 0;
    cudaError_t e = cudaMemcpyFromSymbol(&v, g_tc_abort, sizeof(int));
    if (e != cudaSuccess) return (int)e;
    e = cudaMemcpyToSymbol(g_tc_abort, &zero, sizeof(int));
    if (e != cudaSuccess) return (int)e;
    if (aborted) *aborted = v;
    const int rc = gnm_linear_tc_abort_flag(aborted);
    return rc != GNM_OK ? rc : gnm_linear_bwd_tc_abort_flag(aborted);
}

/* Profiling aid: while non-NULL, every tcgen05 aggregation launch writes per-CTA cycle counters to buf
 * (16 int64 per CTA: [0] epilogue role cycles, [1] waiting for accumulators, [2] MMA role cycles, [3] waiting
 * for A stages, [4] waiting for free accumulator slots, [5] producer role cycles, [6] waiting for free stages). */
extern "C" int gnm_aggregate_tc_set_debug(long long* buf) {
    g_tc_dbg_host = buf;
    return GNM_OK;
}
