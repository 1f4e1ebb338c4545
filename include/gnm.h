/*
 * gnm.h - C ABI of libgnm.so: the B200 (sm_100a) kernels behind graph-neural-mapping's GIN
 * message-passing hot path (GIN_InfoMaxReg forward/backward + DGI Discriminator).
 *
 * The reference has no FFI of its own: every FLOP of this path is a PyTorch ATen call made
 * from /root/reference/models/{graphcnn,mlp,discriminator}.py. Each entry point below names
 * the reference lines (file:line under /root/reference) whose arithmetic it replaces; the
 * Python classes in graph_neural_mapping_b200/models/ keep the reference's constructor and
 * forward signatures and call these through ctypes (see INTEGRATION.md).
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless marked host;
 *   - no hidden allocation, no internal synchronisation, no global state (except the explicitly named A/B switches,
 *     status flags and the gnm_p2p_* buffers): work is enqueued
 *     on `stream` (a cudaStream_t passed as void*, e.g. torch.cuda.current_stream().cuda_stream)
 *     and the call returns immediately;
 *   - return 0 on success, a negative GNM_ERR_* for rejected arguments, or a positive
 *     cudaError_t if the launch failed. Never throws, never falls back to the CPU;
 *   - matrices are fp32 row-major with an explicit leading dimension in ELEMENTS;
 *   - "nullable" pointers may be NULL to disable the corresponding fused step.
 */
#ifndef GNM_H_
#define GNM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNM_OK 0
#define GNM_ERR_BAD_ARG (-1)
#define GNM_ERR_TOO_LARGE (-2)
#define GNM_ERR_ALIGN (-3)

#define GNM_ABI_VERSION 27

typedef void* gnm_stream_t;

/* Peer-memory communicator of the data-parallel step (one process per GPU, GPUs of one NVLink / NVSwitch domain).
 * Host-side POD; peers / counter are DEVICE pointers: peers[world] = every rank's exchange buffer (gnm_p2p_alloc on its
 * owner, gnm_p2p_open elsewhere) as mapped in this process, counter = this rank's call counter (zero-initialised
 * uint32). NULL (or world <= 1) wherever a `const gnm_p2p_comm*` is taken means "single process". */
typedef struct gnm_p2p_comm {
    void* const* peers;
    unsigned int* counter;
    int rank;
    int world;
} gnm_p2p_comm;
#define GNM_P2P_MAX_WORLD 16
#define GNM_P2P_MAX_DOUBLES 256
#define GNM_P2P_HANDLE_BYTES 64

/* BatchNorm finalisation folded into the kernel that PRODUCES the batch statistics ("tail"): host-side POD passed by
 * pointer (nullable = no tail) to gnm_linear / gnm_aggregate_dense_table (forward sums -> gnm_bn_finalize's outputs) and
 * to gnm_relu_bn_bwd_reduce / gnm_aggregate_dense_relu_bn_bwd / gnm_linear_bwd (backward sums -> gnm_bn_bwd_coeffs' output).
 * The last CTA of the producer to finish does the arithmetic of the separate kernel - including, data parallel, the
 * peer-memory all-reduce of the sums - so 20 few-microsecond kernels per training step, each a serial link between
 * two big ones, leave the launch list. Only the tcgen05 / vectorised producers honour a tail; an entry point that
 * cannot returns GNM_ERR_TOO_LARGE before launching anything when one is passed (call the separate kernel then).
 *   kind FINALIZE: count, gamma, beta (nullable), eps, momentum, running_mean / running_var / num_batches_tracked
 *     (nullable), outputs scale, shift, mean, rstd - exactly gnm_bn_finalize;
 *   kind BWD_COEFFS: count, gamma, inputs mean, rstd, output coef [3 * n_feat] - exactly gnm_bn_bwd_coeffs;
 *   comm: nullable peer-memory communicator; counter: DEVICE uint32, zero on entry, left zero. */
#define GNM_BN_TAIL_FINALIZE 1
#define GNM_BN_TAIL_BWD_COEFFS 2
typedef struct gnm_bn_tail {
    int kind;
    double count;
    const float* gamma;
    const float* beta;
    float eps;
    float momentum;
    float* running_mean;
    float* running_var;
    int64_t* num_batches_tracked;
    float* scale;
    float* shift;
    float* mean;
    float* rstd;
    float* coef;
    const gnm_p2p_comm* comm;
    unsigned int* counter;
} gnm_bn_tail;

int gnm_abi_version(void);
const char* gnm_error_string(int code);
/* Bind this library's CUDA runtime to device `dev` (one process per GPU). */
int gnm_set_device(int dev);
int gnm_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* smem_optin_bytes);
/* Process-wide diagnostic counters (host pointer): out[i] = kernels this library has ENQUEUED so far in family i
 * (a kernel recorded during CUDA-graph capture counts once, its replays are the caller's to count). Families:
 * 0 aggregate (CSR warp-per-row), 1 aggregate (mma.sync dense blocks), 2 aggregate (tcgen05), 3 linear (FFMA),
 * 4 linear (tcgen05), 5 linear_bwd (fused FFMA), 6 linear_bwd dX (tcgen05), 7 linear_bwd dW (tcgen05),
 * 8 linear_wgrad (FFMA), 9 every other kernel, 10 linear_bwd one-pass dX + dW (tcgen05), 11 segment_weighted_colsum,
 * 12 ig_expand, 13 ig_accumulate, 14 ig_attribute, 15 occlusion_expand.
 * Returns the number of families (>= 0) or GNM_ERR_BAD_ARG.
 * Tests use it to prove WHICH kernel family a code path ran; bench.py to count launches. */
int gnm_launch_counts(int64_t* out, int n);
/* Programmatic dependent launch of the persistent tcgen05 kernels (aggregation, Linear forward / dX / dW): off by default
 * (no measurable gain inside a CUDA-graph replay at B = 1024; environment GNM_PDL=1 or this call turn it on). When on, a
 * kernel's CTAs may start on SMs the previous kernel of the stream has vacated and
 * run their set-up - barriers, tensor-memory allocation, WEIGHT planes, lookup tables - before that kernel has finished;
 * every access to activations, statistics or coefficients waits for its completion (griddepcontrol.wait). Contract: a
 * call's weight operand must not be written by the kernel immediately in front of it in the stream. */
int gnm_set_pdl(int enabled);
/* Debugging aid for CUDA-graph capture: *status = 0 (stream not capturing), 1 (capturing), 2 (capture invalidated). */
int gnm_stream_capture_status(gnm_stream_t stream, int* status);

/* ---- adjacency / readout structure ------------------------------------------------------ */

/* graphcnn.py:84-106 (__preprocess_neighbors_sumavepool) + the coalesce that torch.spmm performs
 * (graphcnn.py:154,178): block-diagonal CSR of a batch of B graphs from their edge lists.
 *   edges      int64 [2][E_total]: row 0 sources, row 1 destinations, LOCAL node ids, graph after
 *              graph (torch.cat(edge_mat_list, 1) without the start_idx shift);
 *   edge_off   int64 [B+1] prefix of per-graph edge counts; node_off int32 [B+1] prefix of node counts;
 *   add_self_loops = !learn_eps (graphcnn.py:97-102);
 *   local_cols != 0 keeps column ids local to each graph (graph-store form), else global row ids;
 *   n_max      largest node count in the batch (sizes the shared-memory histogram).
 * Output: rowptr int32 [M+1], colidx int32 [E_total + (add_self_loops ? M : 0)], row-major sorted,
 * duplicates kept (a duplicated edge counts twice, like the summed COO). For duplicate-free input it is
 * bit-identical to Adj_block.coalesce().to_sparse_csr().{crow,col}_indices().
 * status int32 [1]: bit 0 is set if any edge index was outside [0, N_g). */
int gnm_csr_build(const int64_t* edges, int64_t e_total, const int64_t* edge_off, const int32_t* node_off,
                  int n_graphs, int n_max, int add_self_loops, int local_cols,
                  int32_t* rowptr, int32_t* colidx, int32_t* status, gnm_stream_t stream);

/* Batch assembly from the device-resident graph store (replaces re-running graphcnn.py:84-106 and the
 * H2D copy of Adj_block every step): slot b copies the stored local CSR of one graph, shifting row
 * pointers by nnz_off[b] and column ids by node_off[b].
 *   src_rowptr_addr / src_colidx_addr / src_tag_addr: int64 [B] device ADDRESSES of each graph's stored
 *   int32 rowptr (N+1 entries), colidx and (nullable) one-hot tag array.
 *   colidx == NULL gathers row pointers and tags only (195 MB less traffic per step at B=1024, N=400): batches that
 *   run on the dense-block kernels read the stored bitmaps and never touch the batch column indices. */
int gnm_csr_batch_gather(const int64_t* src_rowptr_addr, const int64_t* src_colidx_addr, const int64_t* src_tag_addr,
                         const int32_t* node_off, const int64_t* nnz_off, int n_graphs,
                         int32_t* rowptr, int32_t* colidx, int32_t* tags, gnm_stream_t stream);

/* ---- neighbour aggregation -------------------------------------------------------------- */

/* graphcnn.py:154-161 / :178-182: dst[i] = sum_{j in row i} src[map(j)] (/deg(i) for average)
 *                                          + (1 + *eps) * src[map(i)] when eps != NULL.
 * Also its backward (Adj_block is symmetric): mode 2 scales each gathered row by 1/deg(j), which is
 * the transpose of the average. src_map (nullable int32 [M]) redirects row r to src[src_map[r]]: with
 * src = W1^T and src_map = one-hot tags this is the first GIN layer as a row gather (graphcnn.py:195 +
 * mlp.py:48: X_concat is one-hot, so spmm(Adj, X) @ W1^T == gather-sum of W1^T rows).
 * mode: 0 sum, 1 average (0/0 = NaN for an isolated node, as the reference), 2 transpose-of-average.
 * bias (nullable [n_feat]) is added to every output row (the Linear bias of the layer-0 gather path). */
int gnm_aggregate(const int32_t* rowptr, const int32_t* colidx, int n_rows,
                  const float* src, int64_t ld_src, const int32_t* src_map,
                  float* dst, int64_t ld_dst, int n_feat, int mode, const float* eps, const float* bias,
                  gnm_stream_t stream);

/* Per-graph adjacency bitmaps for the tensor-core aggregation: for every graph of a store chunk, row r of
 * its N x ceil(N/32)-word bitmap (at bitmap + bitmap_off[g], word offsets) gets bit c set for every listed
 * neighbour c (rowptr/colidx: the chunk's CSR with LOCAL column ids from gnm_csr_build). dup_flags[g] is set
 * to 1 if a column repeats within a row (a bitmap cannot hold multiplicity: such graphs stay on the CSR path). */
int gnm_bitmap_build(const int32_t* rowptr, const int32_t* colidx, const int32_t* node_off,
                     const int64_t* bitmap_off, int n_graphs, uint32_t* bitmap, int32_t* dup_flags,
                     gnm_stream_t stream);

/* Same contract as gnm_aggregate (graphcnn.py:154-161 / :178-182 and its transpose), computed per graph as a
 * dense 0/1 block product on the tensor cores: dst_g = A_g . src_g with A_g expanded from the graph's bitmap
 * (bitmap_addr[g]: device address) and src split into three bf16 planes (exact for fp32) with fp32
 * accumulation. rowptr (batch CSR row pointers) supplies the degrees for mode 1 / 2 and may be NULL for mode 0.
 * Needs n_feat % 4 == 0 and 16-byte aligned rows (else GNM_ERR_ALIGN: use gnm_aggregate).
 * impl: 0 = auto (tcgen05/TMEM kernel when every graph has <= 416 nodes, else the mma.sync kernel),
 *       1 = mma.sync kernel, 2 = tcgen05 kernel only (GNM_ERR_TOO_LARGE if it does not fit).
 * BatchNorm + ReLU on load: with bn_scale / bn_shift (nullable, [n_feat] each) src is the PRE-BatchNorm output z of the
 * layer below and the kernel aggregates h = relu(z*bn_scale + bn_shift) - graphcnn.py:162-166's h of that layer, the
 * expression of gnm_bn_relu_readout, so dst is bit-identical to gnm_bn_relu_readout(z -> h) + gnm_aggregate_dense(h)
 * without h ever being written. pooled (nullable, ld_pooled) then also receives that layer's readout
 * (graphcnn.py:225-228: pooled[g] = pool_scale[g] (nullable) * sum of the graph's rows of h), i.e. gnm_bn_relu_readout's
 * pooled output, summed in a different order. tcgen05 kernel only, single pass: n_max <= 416, n_feat <= 64, mode 0, no
 * eps / src_map / bias, impl != 1; GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN otherwise, nothing launched (materialise h with
 * gnm_bn_relu_readout and aggregate it then). */
int gnm_aggregate_dense(const int64_t* bitmap_addr, const int32_t* node_off, const int32_t* rowptr,
                        int n_graphs, int n_max, const float* src, int64_t ld_src, const int32_t* src_map,
                        float* dst, int64_t ld_dst, int n_feat, int mode, const float* eps, const float* bias,
                        int impl, const float* bn_scale, const float* bn_shift, float* pooled, int64_t ld_pooled,
                        const float* pool_scale, gnm_stream_t stream);
/* dst = Agg(cA*dy + cB*z + cC): the aggregation of a BatchNorm-backward result (autograd of graphcnn.py:162-166 feeding
 * the transpose of :154-161 at layer 0) without materialising it - coef = [cA | cB | cC] from gnm_bn_bwd_coeffs is
 * applied to the rows as the tcgen05 kernel loads them. Returns GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN when the batch does
 * not fit that kernel (n_max > 416, odd strides): use gnm_bn_bwd_apply + gnm_aggregate* then. No eps self term
 * (learn_eps models take the two-pass route). */
/* Layer 0 on one-hot inputs when every graph of the batch carries the SAME injective tag sequence (util.py:106-116: one
 * tag per ROI, same ROI order for every subject): z0 = Agg(table[tags]) [+ (1+eps) table[tags]] + bias - graphcnn.py:154-161
 * + the first Linear of mlp.py:48 with X_concat = stacked identities - plus the BatchNorm statistics of z0
 * (out_stats, nullable double[2*n_feat], += [sum | sum of squares] per column) taken in the copy-out. The table rows are
 * converted to tensor-core operands once per CTA and stay resident for all its graphs. tcgen05 kernel only
 * (n_max <= 416, n_feat <= 64, mode 0 / 1): GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN otherwise, nothing launched - use
 * gnm_aggregate_dense + gnm_col_stats then. tags: int32 [n_max], ONE graph's tag sequence; every graph has n_max nodes. */
int gnm_aggregate_dense_table(const int64_t* bitmap_addr, const int32_t* node_off, const int32_t* rowptr, int n_graphs,
                              int n_max, const float* table, int64_t ld_table, const int32_t* tags, float* dst,
                              int64_t ld_dst, int n_feat, int mode, const float* eps, const float* bias, double* out_stats,
                              const gnm_bn_tail* tail, gnm_stream_t stream);

int gnm_aggregate_dense_affine(const int64_t* bitmap_addr, const int32_t* node_off, const int32_t* rowptr, int n_graphs,
                               int n_max, const float* dy, int64_t ld_dy, const float* z, int64_t ld_z, const float* coef,
                               float* dst, int64_t ld_dst, int n_feat, int mode, gnm_stream_t stream);
/* Backward aggregation fused with its consumer (autograd of graphcnn.py:154-166 across two layers): what
 * gnm_aggregate_dense(src -> d_h) followed by gnm_relu_bn_bwd_reduce(z, ..., d_h, ...) computes, with the ReLU mask, the
 * readout / DGI gradient terms and the BatchNorm-backward reduction applied in the aggregation kernel's copy-out, so the
 * aggregated gradient never makes the round trip through HBM. tcgen05 kernel only and n_feat <= 64: returns
 * GNM_ERR_TOO_LARGE / GNM_ERR_ALIGN (nothing launched) otherwise - run the two kernels then. Arguments as in those two. */
int gnm_aggregate_dense_relu_bn_bwd(const int64_t* bitmap_addr, const int32_t* node_off, const int32_t* rowptr, int n_graphs,
                                    int n_max, const float* src, int64_t ld_src, int n_feat, int mode, const float* eps,
                                    const float* z, int64_t ldz, const float* scale, const float* shift, const float* mean,
                                    const float* rstd, const float* d_pooled, int64_t ld_dpooled, const float* pool_scale,
                                    const float* d_score, const float* u, int64_t ldu, const float* d_neg, int64_t ld_dneg,
                                    int n_neg, float* dy, int64_t lddy, double* stats, const gnm_bn_tail* tail, gnm_stream_t stream);
/* *aborted = 1 if a tcgen05 kernel (aggregation or linear) launched since the last call ran into a (bounded) barrier-wait timeout
 * and drained without producing valid output. Synchronises the device; meant for tests / smoke checks. */
int gnm_aggregate_tc_status(int* aborted);
/* Profiling aid: while buf != NULL every tcgen05 aggregation launch writes 16 int64 cycle counters per CTA to buf
 * (device memory, >= 16 * #SMs entries): role cycles and barrier-wait cycles of the epilogue, MMA and producer warps. */
int gnm_aggregate_tc_set_debug(long long* buf);

/* d eps[layer] = sum_i <a[i], b[map(i)]> (autograd of graphcnn.py:161). out: double[1], accumulated. */
int gnm_dot_rows(const float* a, int64_t lda, const float* b, int64_t ldb, const int32_t* b_map,
                 int n_rows, int n_feat, double* out, gnm_stream_t stream);

/* dW1^T[tag[r], :] += g[r, :] : gradient of the gathered table (layer-0 one-hot path).
 * workspace (nullable, workspace_floats >= gnm_scatter_rows_workspace(...)) selects the deterministic two-stage
 * merge (per-CTA partial tiles + fixed-order sum); without it partial tiles are merged with fp32 atomics. */
int gnm_scatter_rows_add(const float* g, int64_t ldg, const int32_t* tags, int n_rows, int n_feat,
                         float* table_grad, int64_t ldt, int n_table_rows, float* workspace,
                         int64_t workspace_floats, gnm_stream_t stream);
int64_t gnm_scatter_rows_workspace(int n_rows, int n_feat, int n_table_rows);
/* Same gradient when every graph of the batch carries the same injective tag sequence tags[0..period) (util.py:106-116
 * gives every subject one tag per ROI in the same ROI order): out[tags[t], :] += sum_k g[k*period + t, :] (tags NULL =
 * identity). A streaming column sum instead of a scatter; deterministic (per-split partial sums in workspace, merged in
 * a fixed order). The CALLER guarantees the precondition; rows whose tag falls outside [0, n_table_rows) are dropped.
 * n_rows % period == 0, n_feat % 4 == 0, 16-byte aligned rows; workspace_floats >= gnm_rows_period_workspace(...). */
int gnm_rows_period_sum(const float* g, int64_t ldg, int n_rows, int n_feat, int period, const int32_t* tags, float* out,
                        int64_t ldo, int n_table_rows, float* workspace, int64_t workspace_floats, gnm_stream_t stream);
int64_t gnm_rows_period_workspace(int n_rows, int n_feat, int period);

/* ---- MLP: Linear + BatchNorm + ReLU ------------------------------------------------------ */

/* mlp.py:48-49 / nn.Linear: y[m, n] = sum_k f(x[m, k]) * W(k, n) + bias[n], with
 * W(k, n) = w[n*ldw + k] (w_is_kn == 0, nn.Linear layout [out, in]) or w[k*ldw + n] (w_is_kn == 1,
 * used for dX = dY @ W). f is the fused BatchNorm-apply + ReLU of the PREVIOUS op:
 * f(x) = max(0, x*in_scale[k] + in_shift[k]) when in_scale != NULL (mlp.py:48, graphcnn.py:163-166).
 * col_stats (nullable double [2*n_out], +=): per-column sum and sum of squares of y, the BatchNorm batch
 * statistics of the NEXT op (mlp.py:48, graphcnn.py:163). */
int gnm_linear(const float* x, int64_t ldx, int n_rows, int n_in,
               const float* w, int64_t ldw, int w_is_kn, const float* bias,
               const float* in_scale, const float* in_shift,
               float* y, int64_t ldy, int n_out, double* col_stats, const gnm_bn_tail* tail, gnm_stream_t stream);

/* gnm_linear implementation switch (process-wide A/B aid; the only global setting of the library):
 * 0 = auto (tcgen05 kernel for n_in, n_out <= 64 and n_rows >= 4096, fp32 FFMA kernel otherwise), 1 = FFMA only,
 * 2 = tcgen05 only, 3 = tcgen05 only with gnm_linear_bwd held to its two-pass kernel pair (without it a 64 x 64 aligned unit
 * takes the one-pass kernel). The tcgen05 kernels keep fp32-level accuracy by exact bf16x3 operand splits (six products). */
int gnm_set_linear_impl(int impl);

/* Weight gradient: dw[o, i] += sum_m dz[m, o] * f(x[m, i]); dbias[o] += sum_m dz[m, o] (nullable).
 * f as in gnm_linear (recompute of the BatchNorm+ReLU activation instead of storing it). */
int gnm_linear_wgrad(const float* dz, int64_t lddz, const float* x, int64_t ldx, int n_rows, int n_out, int n_in,
                     const float* in_scale, const float* in_shift,
                     float* dw, int64_t lddw, float* dbias, gnm_stream_t stream);

/* BatchNorm backward as an affine map of (dy, z): dz = A*dy + B*z + C per channel, coef = [A | B | C] ([3*F]).
 * Training (stats != NULL: sum dy, sum dy*xhat; count = global rows): A = g*rstd, B = -g*rstd^2*m2,
 * C = g*rstd*(rstd*m2*mean - m1), m1 = stats[c]/count, m2 = stats[F+c]/count. Eval (stats == NULL): A = g*rstd.
 * With comm the kernel first all-reduces stats in place over peer memory (stats then holds the global sums). */
int gnm_bn_bwd_coeffs(double* stats, double count, const float* gamma, const float* mean, const float* rstd,
                      float* coef, int n_feat, const gnm_p2p_comm* comm, gnm_stream_t stream);

/* Fused backward of one Linear -> BatchNorm (-> ReLU) unit (autograd of mlp.py:48-49, graphcnn.py:162-166) in one
 * pass over the rows, F_out, F_in <= 64 (GNM_ERR_TOO_LARGE otherwise: use the unfused kernels):
 *   dz = A*dy + B*z + C (coef from gnm_bn_bwd_coeffs);  dw[o,i] += sum_m dz[m,o]*a[m,i];  dbias[o] += sum_m dz[m,o]
 *   a = relu(x*in_scale + in_shift) if in_scale != NULL else x          (the unit's input, recomputed)
 *   dx[m,i] = (sum_o dz[m,o]*w[o,i]) * [a[m,i] > 0]                     (nullable; mask only with in_scale)
 *   stats_in[i] += sum_m dx[m,i];  stats_in[F_in+i] += sum_m dx[m,i]*(x[m,i]-in_mean[i])*in_rstd[i]   (nullable)
 * i.e. dx is already the ReLU-masked gradient at the previous unit's BatchNorm output and stats_in its
 * BatchNorm-backward reduction. Kernels: n_rows >= 4096 on sm_100 - a one-pass tcgen05 kernel (dy, z, x read once) when
 * F_out = F_in = 64, dx is requested and every matrix is 16-byte aligned with a leading dimension divisible by four, else a
 * tcgen05 input-gradient kernel followed by a weight-gradient kernel; the fused fp32 FFMA kernel otherwise. */
int gnm_linear_bwd(const float* dy, int64_t lddy, const float* z, int64_t ldz, const float* coef,
                   const float* x, int64_t ldx, const float* in_scale, const float* in_shift,
                   const float* in_mean, const float* in_rstd, const float* w, int64_t ldw,
                   float* dw, int64_t lddw, float* dbias, float* dx, int64_t lddx, double* stats_in,
                   int n_rows, int n_out, int n_in, const gnm_bn_tail* tail, gnm_stream_t stream);

/* Per-column sum / sum of squares (double [2F], +=) of a [M, F] matrix. */
int gnm_col_stats(const float* x, int64_t ldx, int n_rows, int n_feat, double* col_stats, gnm_stream_t stream);

/* nn.BatchNorm1d training statistics -> per-channel affine (mlp.py:38,48; graphcnn.py:51,163,187):
 * mean = sum/count, var = sumsq/count - mean^2 (biased), rstd = 1/sqrt(var + eps);
 * scale = gamma*rstd, shift = beta - mean*scale; running stats updated with momentum (unbiased variance,
 * count/(count-1)) and *num_batches_tracked += 1 when those pointers are non-NULL.
 * `count` is the GLOBAL row count (all ranks): either the caller all-reduces col_stats first (comm NULL) or the kernel
 * does it in place over peer memory (comm, 2*n_feat <= GNM_P2P_MAX_DOUBLES; see the data-parallel section below). */
int gnm_bn_finalize(double* col_stats, double count, const float* gamma, const float* beta,
                    float eps, float momentum, float* running_mean, float* running_var,
                    int64_t* num_batches_tracked, float* scale, float* shift, float* mean, float* rstd,
                    int n_feat, const gnm_p2p_comm* comm, gnm_stream_t stream);

/* Eval-mode BatchNorm (running statistics) as the same per-channel affine. */
int gnm_bn_eval_affine(const float* running_mean, const float* running_var, const float* gamma, const float* beta,
                       float eps, float* scale, float* shift, float* mean, float* rstd, int n_feat,
                       gnm_stream_t stream);

/* graphcnn.py:163-166 + :229: h = relu(z*scale + shift) written to h (nullable) and summed per graph into
 * pooled[g, :] = pool_scale[g] * sum_{rows of g} h  (graph_pool SpMM, graphcnn.py:109-134,229;
 * pool_scale NULL = sum pooling). pooled is OVERWRITTEN ([B, ld_pooled], already offset to the layer slice). */
int gnm_bn_relu_readout(const float* z, int64_t ldz, int n_rows, int n_feat, const float* scale, const float* shift,
                        float* h, int64_t ldh, const int32_t* node_off, int n_graphs, const float* pool_scale,
                        float* pooled, int64_t ld_pooled, gnm_stream_t stream);

/* Backward of relu(batchnorm(z)), pass 1. Assembles the gradient reaching h from up to four sources,
 *   d_out[r, :]                       (nullable; gradient from the next layer's aggregation)
 * + pool_scale[g] * d_pooled[g, :]    (nullable; readout/heads + DGI summary, graphcnn.py:229-239)
 * + d_score[r] * u[g, :]              (nullable; positive DGI score, discriminator.py:28)
 * + d_neg[r, :] for r < n_neg         (nullable; rows used as DGI negatives, graphcnn.py:241-242)
 * masks it with the ReLU (z*scale+shift > 0), writes dy, and accumulates
 * stats[0:F] += sum dy, stats[F:2F] += sum dy * xhat, xhat = (z - mean)*rstd  (double). */
int gnm_relu_bn_bwd_reduce(const float* z, int64_t ldz, int n_rows, int n_feat,
                           const float* scale, const float* shift, const float* mean, const float* rstd,
                           const float* d_out, int64_t ld_dout,
                           const float* d_pooled, int64_t ld_dpooled, const float* pool_scale,
                           const float* d_score, const float* u, int64_t ldu,
                           const float* d_neg, int64_t ld_dneg, int n_neg,
                           const int32_t* node_off, int n_graphs,
                           float* dy, int64_t lddy, double* stats, const gnm_bn_tail* tail, gnm_stream_t stream);

/* Backward of batchnorm, pass 2 (in place on dy):
 * training: dz = gamma*rstd*(dy - stats_sum/count - xhat*stats_dot/count); eval (stats == NULL): dz = dy*gamma*rstd. */
int gnm_bn_bwd_apply(const float* z, int64_t ldz, int n_rows, int n_feat, const float* mean, const float* rstd,
                     const float* gamma, const double* stats, double count, float* dy, int64_t lddy,
                     gnm_stream_t stream);

/* ---- DGI discriminator ------------------------------------------------------------------- */

/* BatchNorm + ReLU on load (the four entry points below): bn (nullable) = per-layer scale | shift, layer l's scale at
 * bn + l*ld_bn and its shift at bn + l*ld_bn + n_feat. With bn, h_all holds each layer's PRE-BatchNorm output z and
 * every value is read as h = relu(z*scale + shift) - graphcnn.py:162-166, gnm_bn_relu_readout's expression - so the
 * results are bit-identical to the same call on the h that gnm_bn_relu_readout would have written. */

/* Copy rows [0, n_rows) of n_f = cat(hidden_rep, 1) (graphcnn.py:233) into a dense [n_rows, L*F] table:
 * the only rows the "shuffled" negatives ever read (graphcnn.py:198-201,241-242). */
int gnm_gather_nf_rows(const float* h_all, int64_t layer_stride, int n_layers, int n_feat, int64_t ldh,
                       int n_rows, const float* bn, int64_t ld_bn, float* table, gnm_stream_t stream);

/* discriminator.py:19-38 with f_k = nn.Bilinear(n_h, n_h, 1) refactored as sc = <h, u_g> + b, u_g = W c_g:
 *   out[r]     = <n_f[r], u[g(r)]> + *bias                    (sc_1, positives)
 *   out[M + r] = <neg_table[neg_idx[g(r)]], u[g(r)]> + *bias  (sc_2: one row per graph, broadcast)
 * h_all holds the L hidden representations as [L][M, ldh]; n_f[r] is their concatenation. */
int gnm_dgi_score_fwd(const float* h_all, int64_t layer_stride, int n_layers, int n_feat, int64_t ldh, int n_rows,
                      const float* u, const float* neg_table, const int32_t* neg_idx,
                      const int32_t* node_off, int n_graphs, const float* bias, const float* bn, int64_t ld_bn,
                      float* out, gnm_stream_t stream);

/* Backward of the scores wrt u, bias and the negative rows:
 *   s2[g]   = sum_{r in g} d_out[M + r]
 *   du[g]   = sum_{r in g} d_out[r] * n_f[r] + s2[g] * neg_table[neg_idx[g]]
 *   d_bias += sum d_out  (double[1])
 * (the gradient wrt n_f itself is fused into gnm_relu_bn_bwd_reduce via d_score/u/d_neg). */
int gnm_dgi_score_bwd(const float* h_all, int64_t layer_stride, int n_layers, int n_feat, int64_t ldh, int n_rows,
                      const float* d_out, const float* neg_table, const int32_t* neg_idx,
                      const int32_t* node_off, int n_graphs, const float* bn, int64_t ld_bn, float* du, float* s2,
                      double* d_bias, gnm_stream_t stream);

/* gnm_dgi_score_fwd, BCEWithLogits against the targets of main.py:32 (positives 1, negatives 0) and gnm_dgi_score_bwd
 * in ONE pass over n_f, for a training step whose loss is the BCE mean (the gradient of a score is local):
 *   out[r], out[M + r] as gnm_dgi_score_fwd;
 *   d_score[r] = grad_scale * (sigmoid(out[r]) - 1)              (d_logits[:M] of gnm_bce_logits)
 *   du, s2, *d_bias += as gnm_dgi_score_bwd with d_out = [d_score, grad_scale * sigmoid(out[M:])];
 *   *loss_acc += loss_scale * sum_{i < 2M} bce(out[i], y_i).
 * Arguments as in those calls (d_bias, loss_acc: DEVICE double[1], accumulated). out and d_score are bit-identical to the
 * three calls, du and s2 equal to fp32 rounding. n_feat == 64 and n_layers <= 5 only (GNM_ERR_TOO_LARGE otherwise),
 * 16-byte aligned rows (GNM_ERR_ALIGN); nothing is launched then - make the three calls instead. */
int gnm_dgi_score_train(const float* h_all, int64_t layer_stride, int n_layers, int n_feat, int64_t ldh, int n_rows,
                        const float* u, const float* neg_table, const int32_t* neg_idx, const int32_t* node_off,
                        int n_graphs, const float* bias, const float* bn, int64_t ld_bn, float grad_scale,
                        double loss_scale, float* out, float* d_score, float* du, float* s2, double* d_bias,
                        double* loss_acc, gnm_stream_t stream);

/* Standalone Discriminator.forward on materialised tensors (discriminator.py:19-38):
 * out[r] = <h[r], u[r / rows_per_graph]> + *bias (+ s_bias[r] if non-NULL). */
int gnm_rowdot_score(const float* h, int64_t ldh, int n_rows, int n_feat, const float* u, int64_t ldu,
                     int rows_per_graph, const float* bias, const float* s_bias, float* out, gnm_stream_t stream);

/* ---- max pooling over neighbours (graphcnn.py:55-81 `__preprocess_neighbors_maxpool`, :137-143 `maxpool`) --------
 * The reference gathers h through a padded neighbour list whose pads point at a dummy row (column-wise minimum of h
 * over the batch, :139-140) and takes torch.max over dim 1. Here: maximum over the CSR row (it holds the self loop
 * exactly when the reference appends the node itself, learn_eps == False); a row with no entry yields the dummy.
 *   gnm_col_min: packed[f] = min_r (order_key(h[r,f]) << 32 | r), caller presets all-ones: the dummy row and, in the
 *     low word, the row that supplied it (torch.min's gradient target).
 *   gnm_aggregate_max: out[i,f] = max_{j in row i} h[j,f] (+ (1+eps) h[i,f]); argmax[i,f] = that j, or n_rows for the
 *     dummy. Ties keep the lowest column id (they occur at exact zeros behind a ReLU, whose backward masks them).
 *   gnm_aggregate_max_bwd: d_h[j,f] = sum_{i in row j, argmax[i,f] == j} d_out[i,f] (+ (1+eps) d_out[j,f]) - pull form
 *     over the same CSR (symmetric structure, as util.py:99-103 builds it), deterministic; dummy hits go to the
 *     column-minimum row. */
int gnm_col_min(const float* h, int64_t ldh, int n_rows, int n_feat, unsigned long long* packed, gnm_stream_t stream);
int gnm_aggregate_max(const int32_t* rowptr, const int32_t* colidx, int n_rows, const float* h, int64_t ldh, int n_feat,
                      const unsigned long long* col_min, const float* eps, float* out, int64_t ld_out, int32_t* argmax,
                      gnm_stream_t stream);
int gnm_aggregate_max_bwd(const int32_t* rowptr, const int32_t* colidx, int n_rows, const float* d_out, int64_t ld_dout,
                          int n_feat, const int32_t* argmax, const unsigned long long* col_min, const float* eps,
                          float* d_h, int64_t ld_dh, gnm_stream_t stream);

/* ---- the [B, L*F]-sized remainder of a training step (SURVEY 8(f) N2; gnm_train.cu) ---------------------------
 * What main.py:31-41 does around the encoder, as a handful of launches instead of ~110 torch kernels.
 *
 * gnm_heads_ce: graphcnn.py:228-231 + main.py:35 forward AND backward in one pass over g_f [B, L*F]:
 *   c_logit[b,c] = sum_l mask[l,b,c] * (<weights[l][c,:], g_f[b, l*F:(l+1)*F]> + biases[l][c])
 *   (mask nullable [L,B,C] = F.dropout's keep mask scaled by 1/(1-p), drawn by the caller from torch's generator),
 *   *loss_acc += inv_count * sum_b CrossEntropy(c_logit[b], labels[b]) (nn.CrossEntropyLoss, mean: inv_count = 1/B),
 *   d_gf[b, :] = d loss / d g_f, d_weights[l] / d_biases[l] = the head gradients (written, deterministic).
 *   weights / biases / d_weights / d_biases: HOST arrays of n_layers device pointers. workspace: at least
 *   gnm_heads_ce_workspace(...) floats; counter: one zero-initialised uint32 (left zero). L <= 16, C <= 8.
 * gnm_bce_logits: nn.BCEWithLogitsLoss (main.py:17,34) against the targets of main.py:32 (first n_pos rows 1, rest 0):
 *   *loss_acc += loss_scale * sum_i bce(logits[i], y_i); d_logits[i] (nullable) = grad_scale * (sigmoid(logits[i]) - y_i).
 * gnm_small_gemm: C[m,n] = sum_k A(m,k) B(k,n), A(m,k) = a[m*sam + k*sak], B(k,n) = b[k*sbk + n*sbn] (any of NT/TN/NN
 *   without copies) for the Discriminator glue on [B, L*F] operands (graphcnn.py:238-239, discriminator.py:28-29
 *   refactored as u_g = W c_g): sigmoid_a != 0 applies sigmoid to A on load and writes it to a_out (c = sigmoid(g_f),
 *   u = c W^T in one launch); dsig_s != NULL makes the epilogue C = dsig_add (nullable) + acc * s * (1 - s)
 *   (d g_f = d_heads + (du W) c (1 - c)).
 * gnm_dgi_neg_grad: d_neg[j,:] = sum_{g: neg_idx[g] == j} s2[g] * u[g,:], j < n_neg - the gradient reaching the
 *   "shuffled" rows n_f[perm[g]] of graphcnn.py:241-242; rows nobody names are zero. Deterministic.
 * gnm_adam_step: torch.optim.Adam (main.py:39-41,136; defaults: no amsgrad) over a table of n_tensors tensors in one
 *   launch: params / grads HOST arrays of device pointers, numel / state_off HOST int arrays (state_off = offset of the
 *   tensor's moments in the flat exp_avg / exp_avg_sq buffers). step: DEVICE float[2], step[0] = steps done so far
 *   (advanced by the call); lr: DEVICE float[1] (schedulers write it in place: visible to a captured CUDA graph).
 *   Same operation order as torch's capturable implementation; grads are multiplied by grad_scale first (1/world
 *   after a summed all-reduce). loss_out (nullable, DEVICE float[1]) = sum of the n_loss_terms doubles - the step's
 *   loss terms accumulated by gnm_heads_ce / gnm_bce_logits - so that no extra launch forms the loss. */
int gnm_heads_ce_workspace(int n_graphs, int n_layers, int n_feat, int n_classes);
int gnm_heads_ce(const float* g_f, int64_t ldg, int n_graphs, int n_layers, int n_feat, int n_classes,
                 const float* const* weights, const float* const* biases, const float* mask, const int64_t* labels,
                 float inv_count, float* c_logit, double* loss_acc, float* d_gf, int64_t ldd, float* const* d_weights,
                 float* const* d_biases, float* workspace, int64_t workspace_floats, unsigned int* counter,
                 gnm_stream_t stream);
/* The two halves of gnm_heads_ce for callers that compute their own loss on c_logit (the reference's driver does,
 * main.py:35): gnm_heads_fwd writes c_logit only; gnm_heads_bwd takes d loss / d c_logit [B, C] and writes d_gf and the
 * head gradients (same workspace / counter contract as gnm_heads_ce). */
int gnm_heads_fwd(const float* g_f, int64_t ldg, int n_graphs, int n_layers, int n_feat, int n_classes,
                  const float* const* weights, const float* const* biases, const float* mask, float* c_logit,
                  gnm_stream_t stream);
int gnm_heads_bwd(const float* g_f, int64_t ldg, int n_graphs, int n_layers, int n_feat, int n_classes,
                  const float* const* weights, const float* mask, const float* d_logit, float* d_gf, int64_t ldd,
                  float* const* d_weights, float* const* d_biases, float* workspace, int64_t workspace_floats,
                  unsigned int* counter, gnm_stream_t stream);
int gnm_bce_logits(const float* logits, int64_t n, int64_t n_pos, float grad_scale, double loss_scale, double* loss_acc,
                   float* d_logits, gnm_stream_t stream);
int gnm_small_gemm(const float* a, int64_t sam, int64_t sak, const float* b, int64_t sbk, int64_t sbn, float* c,
                   int64_t ldc, int m, int n, int k, int sigmoid_a, float* a_out, int64_t lda_out, const float* dsig_s,
                   int64_t lds, const float* dsig_add, int64_t ldadd, gnm_stream_t stream);
int gnm_dgi_neg_grad(const int32_t* neg_idx, const float* s2, const float* u, int64_t ldu, int n_graphs, int width,
                     float* d_neg, int64_t ldn, int n_neg, gnm_stream_t stream);
int gnm_adam_step(float* const* params, const float* const* grads, const int32_t* numel, const int32_t* state_off,
                  int n_tensors, float* exp_avg, float* exp_avg_sq, float* step, const float* lr, double beta1, double beta2,
                  float eps, float weight_decay, float grad_scale, const double* loss_terms, int n_loss_terms,
                  float* loss_out, gnm_stream_t stream);

/* ---- ROI saliency ----------------------------------------------------------------------------------------------
 * The node average of the saliency maps (graphcnn.py:254-299 averaged over the node axis, as evaluate/
 * plot_saliency_nii.py does before painting ROI volumes) without the [N, D] maps: mean_n (Agg^T dz W1)[n] =
 * (1/n_g) (sum_m w_m dz[m]) W1 with w_m the row sums of the aggregation operator. Per graph g (rows node_off[g] ..
 * node_off[g+1]):
 *   out[g, c] = scale_g * sum_{m in g} w_m * v[m, c],   c < width,   scale_g = 1/n_g (an empty graph yields zeros)
 * v = x (coef NULL), or the BatchNorm-backward affine formed on load as gnm_aggregate_dense_affine forms it: v = cA*x +
 *   cB*z + cC with coef = [cA | cB | cC] ([3*width], gnm_bn_bwd_coeffs' output); z NULL means cB = cC = 0 (eval with
 *   running statistics) and z is not read.
 * w_m = the row sum of the aggregation operator of gnm_aggregate (mode 0 sum / 1 average, eps nullable) as its backward
 *   (mode 0 / 2) applies it: rowptr NULL: 1; mode 0: deg_m (the CSR row length: self loop included, duplicate edges with
 *   their multiplicity) [+ 1 + *eps]; mode 1: 1, or 0 for an isolated node [+ 1 + *eps]. The transpose of the average
 *   gathers nothing from an isolated node, so the forward's 0/0 = NaN does not reach the input gradient through it and
 *   is not invented here; a NaN in v still propagates.
 * Rows are summed in a fixed order (deterministic, no atomics). Vectorised when width and the leading dimensions are
 * multiples of 4 and x, z are 16-byte aligned; any width >= 1 and stride otherwise. */
int gnm_segment_weighted_colsum(const float* x, int64_t ldx, const float* z, int64_t ldz, const float* coef,
                                const int32_t* node_off, int n_graphs, int width, const int32_t* rowptr, int mode,
                                const float* eps, float* out, int64_t ld_out, gnm_stream_t stream);

/* ---- integrated gradients (zero baseline, one-hot layer-0 input) -------------------------------------------------
 * IG of the class score F_c at the one-hot input X: IG[n, d] = X[n, d] * sum_s w_s dF_c/dX (alpha_s X)[n, d]. Layer 0 is
 * linear in X (z0(alpha) = alpha * Agg(X) W1^T + b), so the path points run as a VIRTUAL BATCH that repeats every real
 * graph g (rows node_off[g] .. node_off[g+1], n_g rows; node_off[0] = 0, node_off[n_graphs] = n_rows) `points` times,
 * graph-major: virtual row of (graph g, point s, node i) = points * node_off[g] + s * n_g + i. All three calls sum in a
 * fixed order without atomics (bit-reproducible). Vectorised when width and the leading dimensions are multiples of 4
 * and the row operands 16-byte aligned; any width >= 1 and stride otherwise. Negative sizes return GNM_ERR_BAD_ARG;
 * an empty problem returns GNM_OK with no launch.
 *
 * gnm_ig_expand: layer 0's pre-BatchNorm output at every point from ONE real-batch aggregation p = Agg(X) W1^T (no bias):
 *   z[(g, s, i)] = alpha[s] * p[node_off[g] + i] + bias        c < width; bias ([width]) nullable, alpha [points]
 *   z is [points * n_rows, width]. */
int gnm_ig_expand(const float* p, int64_t ldp, const float* bias, const float* alpha, const int32_t* node_off,
                  int n_graphs, int n_rows, int points, int width, float* z, int64_t ldz, gnm_stream_t stream);
/* gnm_ig_accumulate: the quadrature sum of the points' layer-0 gradients back on the real rows, the eval-mode
 * BatchNorm-backward affine applied on load (cB = cC = 0 with running statistics, so z is not read):
 *   out[r] = (accumulate ? out[r] : 0) + weight * cA o sum_{s < points} dy[(g, s, r - node_off[g])]   r in graph g
 * coef = [cA | ...] (gnm_bn_bwd_coeffs' output; only the first `width` floats are read) nullable: cA = 1. The points
 * are summed in ascending order. accumulate = 1 lets a graph's points be split over several calls. */
int gnm_ig_accumulate(const float* dy, int64_t ldy, const float* coef, const int32_t* node_off, int n_graphs,
                      int n_rows, int points, int width, float weight, int accumulate, float* out, int64_t ld_out,
                      gnm_stream_t stream);
/* gnm_ig_attribute: the node-averaged attribution per ROI from t = Agg^T(accumulated dz) ([n_rows, width], real batch)
 * and the layer-0 table W1^T ([n_table_rows, width]):
 *   a[n] = <t[n], table[tags[n]]>          (the per-row form of gnm_dot_rows with b_map = tags)
 *   out[g, d] = (1/n_g) sum_{n in g, tags[n] = d} a[n]          d < n_table_rows (zeros where no node carries tag d)
 * Duplicate tags within a graph add up, in node order. A tag outside [0, n_table_rows) contributes nothing. An empty
 * graph yields zeros. A non-finite entry in any row t[n] of graph g makes out[g, :] NaN: the full attribution
 * X[n, d] * (t W1)[n, d] is 0 * non-finite = NaN in the columns where X is 0, and the node average carries it. */
int gnm_ig_attribute(const float* t, int64_t ldt, const float* table, int64_t ld_table, int n_table_rows,
                     const int32_t* tags, const int32_t* node_off, int n_graphs, int width, float* out, int64_t ld_out,
                     gnm_stream_t stream);

/* ---- ROI occlusion (zero baseline, one-hot layer-0 input) --------------------------------------------------------
 * Occluding ROI d sets input column d to 0. Layer 0's first Linear output then changes by a rank-1 term, so every
 * occluded copy of a graph is written from ONE real-batch aggregation p = Agg(X) W1^T (no bias):
 *   z[v_node_off[v] + i] = p[m] + bias - c_d[m] * w1t[d]          m = node_off[g] + i, g = v_graph[v], d = v_tag[v]
 *   c_d[m] = s_m * #{n in CSR row m : tags[n] = d} + (eps ? (1 + *eps) * [tags[m] = d] : 0)
 *   s_m = 1 (mode 0: sum, and max pooling where it equals the sum), 1 / (rowptr[m+1] - rowptr[m]) (mode 1: average)
 * for every virtual graph v < n_virtual and node i < n_g of its real graph g (rows node_off[g] .. node_off[g+1] of the
 * real batch; the virtual batch's v_node_off[v+1] - v_node_off[v] must equal n_g). rowptr / colidx (GLOBAL column ids)
 * / tags describe the real batch, whose adjacency must be symmetric (the CSR rows of the nodes tagged d then list
 * exactly the rows with a non-zero count). v_tag[v] < 0 or >= n_table_rows makes v a baseline copy: z = p + bias.
 * A row whose c_d[m] is 0 is written as exactly p + bias, so baseline rows and unaffected rows are bit-identical across
 * copies; s_m is formed only for a non-zero count, so an isolated row's 0/0 never multiplies a zero count. Counts are
 * integer adds (exact in any order) and no atomics touch z: bit-reproducible. One CTA per virtual graph; n_max (the
 * largest n_g) above 4096 returns GNM_ERR_TOO_LARGE. bias ([width]) and eps ([1]) nullable; w1t is [n_table_rows,
 * width]. Vectorised when width and the leading dimensions are multiples of 4 and p, z, bias, w1t 16-byte aligned; any
 * width >= 1 and stride otherwise. Negative sizes or a mode other than 0 / 1 return GNM_ERR_BAD_ARG; an empty problem
 * (n_virtual, width or n_max 0) returns GNM_OK with no launch. */
int gnm_occlusion_expand(const float* p, int64_t ldp, const float* bias, const float* w1t, int64_t ld_w1t,
                         int n_table_rows, const int32_t* rowptr, const int32_t* colidx, const int32_t* tags,
                         const int32_t* node_off, int n_graphs, int n_max, const int32_t* v_graph, const int32_t* v_tag,
                         const int32_t* v_node_off, int n_virtual, int width, int mode, const float* eps, float* z,
                         int64_t ldz, gnm_stream_t stream);

/* ---- data parallel: synchronised BatchNorm sums over NVLink peer memory ------------------------------
 * The reference is single-process; a global-batch BatchNorm needs the per-channel sums of all ranks before the next
 * operator can run (20 exchanges per training step, each on the critical path). Instead of an NCCL launch per exchange
 * the CONSUMING kernel does it: gnm_bn_finalize / gnm_bn_bwd_coeffs take a communicator and all-reduce their double[2F]
 * input in place (remote stores into every peer's exchange buffer, system-scope release/acquire flags, fixed-order
 * sum: bit-identical on all ranks) before using it. gnm_p2p_allreduce is the same exchange as a kernel of its own
 * (n <= GNM_P2P_MAX_DOUBLES). All ranks must issue the same sequence of exchanges. Waits are bounded (~10 s):
 * gnm_p2p_status reports a give-up. */
int64_t gnm_p2p_buffer_bytes(void);
int gnm_p2p_alloc(void** buf, unsigned char* handle /* [GNM_P2P_HANDLE_BYTES] out: CUDA IPC handle */);
/* Larger peer-mapped regions for the two bulk exchanges of the data-parallel step - the rows of n_f that the DGI
 * negatives read (graphcnn.py:241-242: rows perm[g] < B_global, all owned by rank 0) with their gradient, and the flat
 * parameter gradients. gnm_p2p_alloc_bytes = gnm_p2p_alloc with a caller-chosen size (zero-filled; opened / closed
 * with gnm_p2p_open / gnm_p2p_close). The data kernels read / write peer memory through ordinary pointers (e.g. the
 * `neg_table` of gnm_dgi_score_fwd may point into rank 0's region); ordering between ranks comes from a
 * gnm_p2p_allreduce of one dummy value used as a barrier (every rank passes it only after all ranks reached it).
 *   gnm_p2p_push: every region r receives src[0..n) at byte_offset (regions: DEVICE array of `world` base pointers as
 *     mapped in this process) - the all-gather half of the gradient all-reduce;
 *   gnm_sum_slots: out = scale * sum_{r < world} base[r*stride .. r*stride + n) in rank order - the reduce half
 *     (bit-identical on every rank); stride a multiple of 4 floats, 16-byte aligned pointers;
 *   gnm_scatter_scaled_rows: dst[idx[g], :] = scale[g] * src[g, :] for injective idx (entries outside [0, n_dst) are
 *     skipped) - each rank writes the gradient rows its permutation slice names straight into rank 0's region. */
int gnm_p2p_alloc_bytes(void** buf, unsigned char* handle, int64_t bytes);
int gnm_p2p_push(const float* src, int64_t n, void* const* regions, int world, int64_t byte_offset, gnm_stream_t stream);
int gnm_sum_slots(const float* base, int world, int64_t stride, int64_t n, float scale, float* out, gnm_stream_t stream);
int gnm_scatter_scaled_rows(const int32_t* idx, const float* scale, const float* src, int64_t lds, int n_src, int width,
                            float* dst, int64_t ldd, int n_dst, gnm_stream_t stream);
int gnm_p2p_open(const unsigned char* handle, void** buf);
int gnm_p2p_close(void* buf, int owner);
int gnm_p2p_allreduce(double* data, int n, const gnm_p2p_comm* comm, gnm_stream_t stream);
int gnm_p2p_status(int* aborted);

#ifdef __cplusplus
}
#endif
#endif /* GNM_H_ */
