/*
 * sldm_sage.h -- C-ABI of the B200-native SageBlock hot path (libsldm_sage.so).
 *
 * This is the drop-in boundary of the repo.  Every entry point takes plain
 * pointers and sizes (no torch types) and launches hand-written sm_100a CUDA
 * kernels on the stream it is given; nothing here synchronises the host unless
 * the comment on the function says so.  The Python host (sldm_gnn_b200/) binds
 * these with ctypes; INTEGRATION.md shows the stub a maintainer of the
 * reference would add.
 *
 * What each group replaces in the reference (paths relative to the reference
 * checkout; PyG = torch-geometric 2.7.0, pinned in uv.lock:1406-1407):
 *
 *   sldm_csr_*            the implicit "index by edge_index[1]" of PyG
 *                         utils/_scatter.py::scatter as called from
 *                         src/models/blocks/sageblock.py:18 (conv(x, edge_index));
 *                         edge_index contract: src/models/grusage.py:153,182 and
 *                         src/gbuilder.py:88-112 (int64 [2,E], row 0 = source,
 *                         row 1 = destination).
 *   sldm_segment_mean     MessagePassing.propagate + MeanAggregation
 *                         (x.index_select(0, edge_index[0]) then
 *                         scatter(reduce='mean') by edge_index[1]).
 *   sldm_sage_project_*   SAGEConv.forward's lin_l(agg) + lin_r(x) followed by
 *                         posts[i] = LayerNorm -> LeakyReLU|ReLU
 *                         (src/models/blocks/sageblock.py:10-14,18-19).
 *   sldm_sage_layer_*     one whole iteration of the loop at
 *                         src/models/blocks/sageblock.py:17-19 (dropout excluded:
 *                         it stays torch's, SURVEY F10), forward and backward.
 *   sldm_gru_*            the sequence head in front of the block: nn.GRU's last
 *                         hidden state (src/models/grusage.py:55-60,160-161).
 *   sldm_sage_block_*_host  the whole SageBlock.forward
 *                         (src/models/blocks/sageblock.py:16-20) for hosts that
 *                         own no device memory: host buffers in, host buffers out.
 *
 * Conventions
 *   - all feature matrices are row-major fp32, contiguous; weights are
 *     [Fout, Fin] row-major exactly as torch.nn.Linear / PyG Linear store them;
 *   - all pointers are DEVICE pointers unless the name ends in _host / _h;
 *   - return value: SLDM_OK or an SLDM_E* code; sldm_last_error() gives the
 *     message for the calling thread;
 *   - sldm_stream_t is a cudaStream_t passed as void* (0 = legacy default);
 *   - indices: the CSR object is int32 (N and E must be < 2^31 - 2^20).
 */
#ifndef SLDM_SAGE_H_
#define SLDM_SAGE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLDM_ABI_VERSION 1

#define SLDM_OK            0
#define SLDM_EINVAL        1  /* bad argument value (Python host: ValueError)   */
#define SLDM_ESHAPE        2  /* inconsistent sizes (Python host: RuntimeError) */
#define SLDM_ECUDA         3  /* CUDA runtime / launch failure                  */
#define SLDM_EWORKSPACE    4  /* workspace too small                            */
#define SLDM_EUNSUPPORTED  5  /* size outside what the kernels cover            */
#define SLDM_ENODEVICE     6  /* no CUDA device: there is no CPU fallback       */

typedef void* sldm_stream_t;

/* ---- library ------------------------------------------------------------ */
int         sldm_abi_version(void);
const char* sldm_last_error(void);
/* kernels launched by this library since it was loaded (bench.py's gpu_launches) */
int64_t     sldm_launch_count(void);
/* number of SMs of the current device (host sync-free after the first call) */
int         sldm_device_sm_count(int* out_sms);

/* ---- CSR object ----------------------------------------------------------
 * One int32 device buffer holding, at the offsets sldm_csr_layout() reports:
 *   meta[64]         [0] hub chunks (by dst)  [1] hub chunks (by src)
 *                    [2] 1 if any index was outside [0,N)   (then clamped)
 *                    [3] 1 if edge_index[0] is NOT non-decreasing
 *                    [4] 1 if edge_index[1] is NOT non-decreasing
 *   rowptr_dst[N+1]  in-edges of node i are col_src[rowptr_dst[i]..rowptr_dst[i+1])
 *   col_src[E]       source ids, STABLE in edge order inside every segment
 *   rowptr_src[N+1]  out-edges (transpose CSR, used by backward)
 *   col_dst[E]       destination ids, stable in edge order inside every segment
 *   hub_dst[cap*4]   work list {row, chunk, nchunks, first_slot} for rows whose
 *   hub_src[cap*4]   degree exceeds SLDM_HUB_DEGREE (split deterministically)
 * Bit-exact contract: rowptr == cumsum(bincount(idx, N)), col == other[argsort(idx, stable)].
 */
#define SLDM_HUB_DEGREE 256   /* rows with more in-edges than this are split   */
#define SLDM_HUB_CHUNK  2048  /* edges per split piece                         */

enum {
  SLDM_CSR_META = 0, SLDM_CSR_ROWPTR_DST = 1, SLDM_CSR_COL_SRC = 2,
  SLDM_CSR_ROWPTR_SRC = 3, SLDM_CSR_COL_DST = 4, SLDM_CSR_HUB_DST = 5,
  SLDM_CSR_HUB_SRC = 6, SLDM_CSR_TOTAL = 7
};
/* offsets (in int32 elements) of the 7 sections; out8[SLDM_CSR_TOTAL] = total size */
int     sldm_csr_layout(int64_t N, int64_t E, int64_t* out8);
int64_t sldm_csr_workspace_bytes(int64_t N, int64_t E);
/* edge_index: device int64 [2,E] contiguous.  Never written.  E == 0 is legal. */
int     sldm_csr_build(const int64_t* edge_index, int64_t E, int64_t N,
                       int32_t* csr, void* workspace, int64_t workspace_bytes,
                       sldm_stream_t stream);

/* Deferred range report: copies meta[2] of a built CSR object into *status_host_pinned (page-locked host memory the
 * caller preset to -1) behind the build on `stream`, without synchronising: 0 = all indices in range, 1 = some index
 * was outside [0, N) (the reference stack raises IndexError / a device assert there; see sldm_gnn_b200/ops.py). */
int     sldm_csr_status_async(const int32_t* csr, int32_t* status_host_pinned, sldm_stream_t stream);

/* Same build from two separate int64 rows.  edge_src == NULL means source ids 0..E-1: the result is then a
 * membership list (row k of rowptr_dst / col_src = the positions e with edge_dst[e] == k, ascending), which is how
 * the graph readout below obtains the nodes of every graph from PyG's `batch` vector.  In that mode N only bounds
 * edge_dst (N = number of graphs) and the transpose sections (rowptr_src, col_dst, hub_src) are not written. */
int     sldm_csr_build_pairs(const int64_t* edge_src, const int64_t* edge_dst, int64_t E, int64_t N,
                             int32_t* csr, void* workspace, int64_t workspace_bytes,
                             sldm_stream_t stream);

/* ---- segment mean (the aggregation alone) --------------------------------
 * out[i,:] = (sum over k in segment i of src[col[k],:]) / max(deg_i,1)   (mean=1)
 * out[i,:] = addend[i,:] + sum ...                                       (mean=0)
 * transpose=0 walks (rowptr_dst,col_src); transpose=1 walks (rowptr_src,col_dst).
 * Summation inside a segment is sequential in edge order (== the CPU scatter_add_
 * order of the reference) for rows of degree <= SLDM_HUB_DEGREE; hub rows are
 * split in fixed pieces and recombined in piece order (deterministic).
 */
int64_t sldm_segment_workspace_bytes(int64_t N, int64_t E, int32_t F);
int     sldm_segment_reduce(const float* src, int64_t N, int32_t F,
                            const int32_t* csr, int64_t E, int32_t transpose,
                            int32_t mean, const float* addend, float* out,
                            void* workspace, int64_t workspace_bytes,
                            sldm_stream_t stream);

/* ---- projection + LayerNorm + activation ---------------------------------
 * z = agg W_l^T + b_l + x W_r^T ; xhat = (z-mean)*rstd ; y = xhat*g+b ;
 * out = y > 0 ? y : slope*y        (slope = 0 -> ReLU)
 * xhat_out / rstd_out may be NULL (inference).
 */
int64_t sldm_sage_project_workspace_bytes(int64_t N, int32_t Fin, int32_t Fout);
int     sldm_sage_project_forward(const float* agg, const float* x, int64_t N,
                                  int32_t Fin, int32_t Fout,
                                  const float* W_l, const float* b_l, const float* W_r,
                                  const float* ln_w, const float* ln_b,
                                  float eps, float slope,
                                  float* out, float* xhat_out, float* rstd_out,
                                  void* workspace, int64_t workspace_bytes,
                                  sldm_stream_t stream);

/* ---- one SageBlock layer --------------------------------------------------
 * forward : agg = segment_mean(x); out = act(LN(agg W_l^T + b_l + x W_r^T))
 *           agg is always written ([N,Fin]; it is the saved tensor in training
 *           and scratch in inference); xhat/rstd only when non-NULL.
 * backward: given dout = dL/dout, produces dx (may be NULL: not needed),
 *           dW_l, db_l, dW_r, dln_w, dln_b (overwritten, not accumulated).
 *           dz [N,Fout], dagg [N,Fin] and dxroot [N,Fin] are caller-provided
 *           scratch (dagg/dxroot may be NULL iff dx is NULL).
 */
int64_t sldm_sage_layer_fwd_workspace_bytes(int64_t N, int64_t E, int32_t Fin, int32_t Fout);
int     sldm_sage_layer_forward(const float* x, int64_t N, int32_t Fin, int32_t Fout,
                                const int32_t* csr, int64_t E,
                                const float* W_l, const float* b_l, const float* W_r,
                                const float* ln_w, const float* ln_b,
                                float eps, float slope,
                                float* out, float* agg, float* xhat_out, float* rstd_out,
                                void* workspace, int64_t workspace_bytes,
                                sldm_stream_t stream);

int64_t sldm_sage_layer_bwd_workspace_bytes(int64_t N, int64_t E, int32_t Fin, int32_t Fout);
int     sldm_sage_layer_backward(const float* dout, const float* x, const float* agg,
                                 const float* xhat, const float* rstd,
                                 int64_t N, int32_t Fin, int32_t Fout,
                                 const int32_t* csr, int64_t E,
                                 const float* W_l, const float* W_r,
                                 const float* ln_w, const float* ln_b, float slope,
                                 float* dx, float* dW_l, float* db_l, float* dW_r,
                                 float* dln_w, float* dln_b,
                                 float* dz, float* dagg, float* dxroot,
                                 void* workspace, int64_t workspace_bytes,
                                 sldm_stream_t stream);

/* Profiling entry point: the same backward with a mask of the kernels to launch, so that a caller (bench.py) can time
 * each of them alone with CUDA events.  A stage that is masked out must have run before on the same buffers (dz, dagg,
 * dxroot and the workspace carry its results).  SLDM_BWD_STAGE_ALL == sldm_sage_layer_backward. */
#define SLDM_BWD_STAGE_LN     1   /* LayerNorm / activation backward: dz + column partials (k_ln_bwd_rows)           */
#define SLDM_BWD_STAGE_DGRAD  2   /* dagg = (dz W_l)/count, dxroot = dz W_r (k_sage_tc<MODE_DGRAD>)                 */
#define SLDM_BWD_STAGE_WGRAD  4   /* dW_l, dW_r (k_wgrad_tc) + the fixed-order reductions of all partials           */
#define SLDM_BWD_STAGE_GATHER 8   /* dx = dxroot + transpose segment sum of dagg (k_segment_rows_lean)              */
#define SLDM_BWD_STAGE_ALL    15
int     sldm_sage_layer_backward_stages(const float* dout, const float* x, const float* agg,
                                        const float* xhat, const float* rstd,
                                        int64_t N, int32_t Fin, int32_t Fout,
                                        const int32_t* csr, int64_t E,
                                        const float* W_l, const float* W_r,
                                        const float* ln_w, const float* ln_b, float slope,
                                        float* dx, float* dW_l, float* db_l, float* dW_r,
                                        float* dln_w, float* dln_b,
                                        float* dz, float* dagg, float* dxroot,
                                        void* workspace, int64_t workspace_bytes,
                                        sldm_stream_t stream, int32_t stages);

/* ---- bf16 feature storage (BASELINE.json configs[4]: "fp32 vs bf16 features") ------------------------------------
 * The reference has no reduced-precision mode (no autocast / bfloat16 anywhere: main.py:58, src/utils.py:176-236);
 * this is an addition of this library with its own tolerance, the fp32 entry points above stay the parity path.
 * What is stored as bf16 (2 bytes per feature in HBM): the layer input x, the aggregated rows agg and the layer
 * output out -- i.e. every [N, F] feature matrix the forward moves.  What stays fp32: all parameters, every
 * accumulation (segment sums, the tcgen05 products, LayerNorm statistics), the saved xhat / rstd, and the whole
 * backward data path (dout, dz, dagg, dxroot, dx and the parameter gradients); only the weight-gradient kernel
 * reads the bf16 x / agg.  Rounding happens once per stored value (round-to-nearest-even).
 *   sldm_segment_mean_bf16        src, out: bf16 [N,F]; F % 8 == 0, F <= 256
 *   sldm_sage_project_forward_bf16  agg, x bf16 [N,Fin] -> out bf16 [N,Fout] (the projection + LayerNorm + activation alone)
 *   sldm_sage_layer_forward_bf16  x bf16 [N,Fin]; out bf16 [N,Fout]; agg bf16 [N,Fin]; xhat fp32, rstd fp32 (or NULL)
 *   sldm_sage_layer_backward_bf16 x, agg bf16; everything else as sldm_sage_layer_backward_stages (fp32)
 * Shapes: Fin in {64, 128}, Fout % 32 == 0, 32 <= Fout <= 128 (sldm_sage_bf16_supported); otherwise
 * SLDM_EUNSUPPORTED and the caller converts to fp32.  Workspace sizes are those of the fp32 entry points. */
int sldm_sage_bf16_supported(int32_t Fin, int32_t Fout);
int sldm_segment_mean_bf16(const void* src, int64_t N, int32_t F, const int32_t* csr, int64_t E, void* out,
                           void* workspace, int64_t workspace_bytes, sldm_stream_t stream);
int sldm_sage_project_forward_bf16(const void* agg, const void* x, int64_t N, int32_t Fin, int32_t Fout,
                                   const float* W_l, const float* b_l, const float* W_r,
                                   const float* ln_w, const float* ln_b, float eps, float slope,
                                   void* out, float* xhat_out, float* rstd_out,
                                   void* workspace, int64_t workspace_bytes, sldm_stream_t stream);
int sldm_sage_layer_forward_bf16(const void* x, int64_t N, int32_t Fin, int32_t Fout,
                                 const int32_t* csr, int64_t E,
                                 const float* W_l, const float* b_l, const float* W_r,
                                 const float* ln_w, const float* ln_b, float eps, float slope,
                                 void* out, void* agg, float* xhat_out, float* rstd_out,
                                 void* workspace, int64_t workspace_bytes, sldm_stream_t stream);
int sldm_sage_layer_backward_bf16(const float* dout, const void* x, const void* agg,
                                  const float* xhat, const float* rstd,
                                  int64_t N, int32_t Fin, int32_t Fout,
                                  const int32_t* csr, int64_t E,
                                  const float* W_l, const float* W_r,
                                  const float* ln_w, const float* ln_b, float slope,
                                  float* dx, float* dW_l, float* db_l, float* dW_r,
                                  float* dln_w, float* dln_b,
                                  float* dz, float* dagg, float* dxroot,
                                  void* workspace, int64_t workspace_bytes,
                                  sldm_stream_t stream, int32_t stages);

/* ---- graph readout (the consumer of the SageBlock output) -----------------
 * Replaces global_mean_pool / global_max_pool of PyG 2.7.0 (nn/pool/glob.py -> utils/_scatter.py::scatter with
 * reduce='mean' / 'max') as used at src/models/grusage.py:113-120 (choice) and :185 (x = self.global_pool(x, batch)):
 *   mean[g,:] = sum_{i: batch[i]=g} x[i,:] / max(count_g,1)      max[g,:] = max_{i: batch[i]=g} x[i,:]
 *   empty graph -> 0 in both.  'double' = [mean | max] concatenated: pass the two halves of one [G,2F] buffer, ld = 2F.
 * csr is the membership CSR: sldm_csr_build_pairs(NULL, batch, N, csr_nodes >= G, ...), so `batch` need not be
 * sorted.  backward: dx[i,:] = dmean[g,:]/max(count_g,1) + [x[i,:]==max[g,:]] * dmax[g,:]/ties[g,:]  (torch's amax
 * backward shares the gradient evenly among tied maxima).  Either output / gradient view may be NULL.
 */
int64_t sldm_readout_workspace_bytes(int64_t G, int32_t F);
int     sldm_readout_forward(const float* x, int64_t N, int32_t F, const int32_t* csr, int64_t csr_nodes,
                             int64_t G, float* out_mean, float* out_max, int64_t ld, sldm_stream_t stream);
int     sldm_readout_backward(const float* x, int64_t N, int32_t F, const int64_t* batch,
                              const int32_t* csr, int64_t csr_nodes, int64_t G,
                              const float* out_max, int64_t ld_max,
                              const float* dmean, const float* dmax, int64_t ld_d,
                              float* dx, void* workspace, int64_t workspace_bytes, sldm_stream_t stream);

/* ---- mini-batch assembly (the producer of the SageBlock input) -------------
 * Replaces torch_geometric.data.Batch.from_data_list / collate (PyG 2.7.0) as used by the reference's DataLoader
 * (main.py:166-167, src/utils.py:218-223) for graphs that already live on the device (src/dataset.py:75-89):
 *   sldm_concat_chunks       out[dst_off_g .. +bytes_g) = src_g[0 .. bytes_g): torch.cat along dim 0 of G tensors.
 *                            table_dev: G rows of four int64 {src device pointer, dst byte offset, byte count, 0}.
 *   sldm_collate_graph_index edge_index_out[:, eoff_g + k] = edge_index_g[:, k] + node_ptr[g]  (int64 [2, Etot]) and
 *                            batch_out[i] = g for node_ptr[g] <= i < node_ptr[g+1] (may be NULL).
 *                            table_dev: G rows {edge_index_g device pointer, eoff_g, e_g, row stride in elements}.
 * At most 65535 graphs per call; max_* size the grids (largest chunk).  Bit-exact by construction.
 */
int sldm_concat_chunks(const void* table_dev, int64_t G, int64_t max_chunk_bytes, void* out, sldm_stream_t stream);
int sldm_collate_graph_index(const void* table_dev, const int64_t* node_ptr_dev, int64_t G, int64_t Etot,
                             int64_t max_edges, int64_t max_nodes, int64_t* edge_index_out,
                             int64_t* batch_out, sldm_stream_t stream);

/* ---- map attention (between the map-graph block and the vehicle-graph block) --
 * Replaces MapSpatialAttention.forward, src/models/map/mapattention.py:21-56 (called at src/models/grusage.py:175-178):
 *   dist[b,s] = ||pos_b - centroid_s||_2 ; the K nearest segments (ties: lower index first) ;
 *   score_k = W2 . relu(W1 * dist_k + b1) + b2   (attn_mlp = Linear(1,H) -> ReLU -> Linear(H,1); W1, b1, W2 are [H]) ;
 *   w = softmax_k(score) ; ctx[b,:] = sum_k w_k emb[idx_k,:].
 * forward also returns idx [B,K] int64 (ascending distance), dist [B,K], w [B,K] (the saved tensors of backward).
 * backward: gradients for emb (demb [S,D], may be NULL) and the four MLP tensors; positions and centroids are data.
 * csr = membership CSR of idx: sldm_csr_build_pairs(NULL, idx, B*K, csr_nodes >= S, ...) (only needed for demb).
 * K <= 32 (sldm_map_attention_max_k()), H <= 64, S >= K (else SLDM_ESHAPE, like torch.topk).  K <= 8 and K > 8 run
 * different kernels (a per-thread sorted list up to 8, one warp per position above) under the same contract.
 * Backward workspace: sldm_map_attention_workspace_bytes_k(B, H, K); sldm_map_attention_workspace_bytes(B, H) is the
 * same size for any K <= 8.  K > 8 also needs B * K < 2^31 - 2^20 (the membership CSR).
 * Two forward entry points with identical results (bit for bit):
 *   sldm_map_attention_forward       exhaustive scan of the S centroids per position (no preparation);
 *   sldm_map_attention_forward_grid  ring search over a uniform grid of the centroids.  The centroids are a constant
 *                                    of the reference module (register_buffer, mapattention.py:9), so the grid is built
 *                                    once per map: sldm_map_grid_build(centroids, S, grid, sldm_map_grid_bytes(S), ..)
 *                                    and reused by every forward; rebuild it when the centroids change.
 * Non-finite positions or centroids: memory-safe, selection unspecified.
 */
int64_t sldm_map_attention_workspace_bytes(int64_t B, int32_t H);
int64_t sldm_map_attention_workspace_bytes_k(int64_t B, int32_t H, int32_t K);
int     sldm_map_attention_max_k(void);
int64_t sldm_map_grid_bytes(int64_t S);
int     sldm_map_grid_build(const float* centroids, int64_t S, void* grid, int64_t grid_bytes, sldm_stream_t stream);
int     sldm_map_attention_forward_grid(const float* pos, int64_t B, const void* grid, int64_t grid_bytes, int64_t S,
                                        const float* emb, int32_t D, int32_t K,
                                        const float* W1, const float* b1, const float* W2, const float* b2, int32_t H,
                                        float* ctx, int64_t* idx_out, float* dist_out, float* w_out,
                                        sldm_stream_t stream);
int     sldm_map_attention_forward(const float* pos, int64_t B, const float* centroids, int64_t S,
                                   const float* emb, int32_t D, int32_t K,
                                   const float* W1, const float* b1, const float* W2, const float* b2, int32_t H,
                                   float* ctx, int64_t* idx_out, float* dist_out, float* w_out,
                                   sldm_stream_t stream);
int     sldm_map_attention_backward(const float* dctx, int64_t B, const float* emb, int64_t S, int32_t D, int32_t K,
                                    const int64_t* idx, const float* dist, const float* w,
                                    const float* W1, const float* b1, const float* W2, int32_t H,
                                    const int32_t* csr, int64_t csr_nodes,
                                    float* demb, float* dW1, float* db1, float* dW2, float* db2,
                                    void* workspace, int64_t workspace_bytes, sldm_stream_t stream);

/* ---- proximity edges between trajectories (the producer of edge_index) -----
 * Replaces the O(V^2 T) Python double loop of src/gbuilder.py:88-112 / :244-268 (GraphOnlineCreator, rcv.py:77):
 * x is [V, T, F] fp32 (feature 0 = X, 1 = Y, 4 = presence flag); for every ordered pair i != j the distances over the
 * frames where both are present give an edge iff their minimum is <= m_radius, with attributes
 * [min, max, mean, mean of squares]; edges come out in (i, j) lexicographic order like the reference's lists.
 *   count: counts[V], offsets[V+1]; the caller reads E = offsets[V] (device -> host) to size the outputs,
 *   fill : edge_index int64 [2,E], edge_attr fp32 [E,4].      T <= 128.
 */
int sldm_edge_build_count(const float* x, int64_t V, int32_t T, int32_t F, float m_radius,
                          int32_t* counts, int32_t* offsets, sldm_stream_t stream);
int sldm_edge_build_fill(const float* x, int64_t V, int32_t T, int32_t F, float m_radius,
                         const int32_t* offsets, int64_t E, int64_t* edge_index, float* edge_attr,
                         sldm_stream_t stream);

/* ---- sequence head: fused GRU layers, last hidden state ----------------------
 * Replaces `gru_out, hlast = self.gru(x); x = hlast[-1]` (src/models/grusage.py:160-161; nn.GRU(input_size = dynamic
 * features, hidden_size, num_layers = 1, batch_first = True) built at grusage.py:55-60, h0 = 0) and its autograd
 * backward.  x [N,T,I] fp32 contiguous; W_ih [3H,I], W_hh [3H,H] (16-byte aligned), b_ih, b_hh [3H]: torch's
 * weight_ih_l0 / weight_hh_l0 / bias_ih_l0 / bias_hh_l0, gates ordered (r, z, n).  Same formulas as ATen's fused cell.
 *   supported: H in {32, 64, 96}, I <= 8, T*I small enough for the shared-memory tile (sldm_gru_supported() != 0);
 *              anything else returns SLDM_EUNSUPPORTED (the host module then takes the projected path below, or
 *              keeps torch's library GRU).
 *   forward  : h_last [N,H].  Training: saved [T,N,5,H] (NULL for inference) receives, per step and sequence,
 *              h_{t-1} | r | z | n | W_hn h + b_hn -- what backward needs (time-major so that a tile's stores of one
 *              step are contiguous).
 *   backward : dh_last [N,H] in; dgh [T,N,3H] = gradients of the hidden-side gate pre-activations (input of
 *              sldm_gru_wgrad); dgi_n [T,N,H]
 *              (NULL unless dx is wanted: the input-side pre-activation gradients are [dgh[..., :2H] | dgi_n]);
 *              partials [sldm_gru_partial_rows(N)][sldm_gru_partial_width(H)]: per-tile sums the caller adds over
 *              rows, laid out as [28*H/32][32]: v = (u*3+g)*8 + i -> dW_ih[g*H + 32u + lane][i]; v = 24U + u*3 + g ->
 *              db_ih[g*H + 32u + lane]; v = 27U + u -> db_hh[2H + 32u + lane] (db_hh[:2H] = db_ih[:2H]), U = H/32.
 *   wgrad    : dW_hh = dgh^T . h_prev over the T*N rows (h_prev read in place from `saved`), as
 *              sldm_gru_wgrad_tiles(N, T) partial [3H,H] tiles (one per persistent CTA) the caller adds up.
 *
 * Stacked layers (nn.GRU(num_layers = L), no inter-layer dropout): layer l >= 1 reads the output sequence h^{l-1}_t of
 * the layer below, W_ih_l is [3H,H]; only the last step of the last layer is consumed.  All sequence buffers are
 * time-major: h_seq [T,N,H], gi / dgi [T,N,3H], dh_seq [T,N,H].  Per layer l >= 1:
 *   forward  : sldm_gru_project_forward(h_seq^{l-1} -> gi), then sldm_gru_layer_forward with gi (x = NULL).
 *   backward : sldm_gru_layer_backward (x = NULL, dh_seq = the gradient of h^l_t from the layer above or NULL,
 *              dh_last NULL below the top) -> dgh, dgi; dW_hh by sldm_gru_wgrad; dW_ih by
 *              sldm_gru_wgrad_strided(dgi, h_seq^{l-1}, stride H); the layer below's dh_seq by
 *              sldm_gru_project_backward(dgi -> dY).
 *   Layer 0 is the single-layer path plus h_seq (forward) and dh_seq (backward).
 *   stack_supported : layer 0 within sldm_gru_supported(T, I, H); the layers above have no T limit.
 *   layer_forward   : exactly one of x [N,T,I] (layer 0: W_ih [3H,I], b_ih used) or gi [T,N,3H] (16-byte aligned,
 *                     b_ih included; W_ih, b_ih, I ignored).  h_last [N,H] may be NULL; saved as above (NULL for
 *                     inference); h_seq [T,N,H] receives h_t of every step (NULL: not written).
 *   layer_backward  : x NULL selects the deep mode (I ignored; the dW_ih slots of the partials are zeros, the bias
 *                     slots as above).  dh_last [N,H] may be NULL (zeros); dh_seq [T,N,H] may be NULL; dgi_n as
 *                     above; dgi [T,N,3H] (may be NULL) receives the input-side pre-activation gradients [dr dz dn].
 *   project_forward : gi[r] = b_ih + h_seq[r] . W_ih^T over rows = T*N ([H] -> [3H]); project_backward:
 *                     dy[r] = dgi[r] . W_ih ([3H] -> [H]).  W_ih [3H,H]; inputs 16-byte aligned.  FP32 FMA chains in
 *                     sequential k order.
 *   wgrad_strided   : sldm_gru_wgrad with the second operand's row stride given (a multiple of 4, >= H): 5H reads
 *                     h_prev in place from `saved` (= sldm_gru_wgrad), H reads an h_seq (dW_ih = dgi^T . h_seq).
 *
 * Projected layer 0 (sequences too long or inputs too wide for the x tile above): layer 0 is fed like the layers
 * above it, through gi, so neither T nor the tile limits it.
 *   projected_supported   : H in {32, 64, 96} and 1 <= I <= 128 (W_ih is held in shared memory); no limit on T.
 *   input_project_forward : gi[t][n][:] = b_ih + W_ih . x[n][t][:], x [N,T,I] batch-first -> gi [T,N,3H] time-major;
 *                           then sldm_gru_layer_forward with gi.  W_ih [3H,I].  FP32 FMA chains in sequential k
 *                           order, starting from the bias.
 *   backward              : sldm_gru_layer_backward in the deep mode (x = NULL) -> dgh, dgi and the bias partials;
 *                           dW_hh by sldm_gru_wgrad; dW_ih by sldm_gru_input_wgrad.
 *   input_wgrad           : dW_ih [3H,I] = sum over the T*N rows of dgi[t][n]^T . x[n][t], as the first
 *                           sldm_gru_wgrad_tiles(N, T) partial [3H,I] tiles of `partials` (the caller adds them up; a
 *                           fixed order, so the sum is the same run to run).  dgi 16-byte aligned.
 */
int     sldm_gru_supported(int32_t T, int32_t I, int32_t H);
int     sldm_gru_stack_supported(int32_t T, int32_t I, int32_t H);
int64_t sldm_gru_partial_rows(int64_t N);
int64_t sldm_gru_partial_width(int32_t H);
int     sldm_gru_forward(const float* x, int64_t N, int32_t T, int32_t I, int32_t H,
                         const float* W_ih, const float* W_hh, const float* b_ih, const float* b_hh,
                         float* h_last, float* saved, sldm_stream_t stream);
int     sldm_gru_layer_forward(const float* x, const float* gi, int64_t N, int32_t T, int32_t I, int32_t H,
                               const float* W_ih, const float* W_hh, const float* b_ih, const float* b_hh,
                               float* h_last, float* saved, float* h_seq, sldm_stream_t stream);
int     sldm_gru_backward(const float* x, int64_t N, int32_t T, int32_t I, int32_t H, const float* W_hh,
                          const float* dh_last, const float* saved, float* dgh, float* dgi_n, float* partials,
                          int64_t partial_rows, sldm_stream_t stream);
int     sldm_gru_layer_backward(const float* x, int64_t N, int32_t T, int32_t I, int32_t H, const float* W_hh,
                                const float* dh_last, const float* dh_seq, const float* saved, float* dgh,
                                float* dgi_n, float* dgi, float* partials, int64_t partial_rows, sldm_stream_t stream);
int     sldm_gru_project_forward(const float* h_seq, int64_t rows, int32_t H, const float* W_ih, const float* b_ih,
                                 float* gi, sldm_stream_t stream);
int     sldm_gru_project_backward(const float* dgi, int64_t rows, int32_t H, const float* W_ih, float* dy,
                                  sldm_stream_t stream);
int64_t sldm_gru_wgrad_tiles(int64_t N, int32_t T);
int     sldm_gru_wgrad(const float* dgh, const float* saved, int64_t N, int32_t T, int32_t H,
                       float* partials, int64_t partial_tiles, sldm_stream_t stream);
int     sldm_gru_wgrad_strided(const float* dg, const float* a, int64_t a_stride, int64_t N, int32_t T, int32_t H,
                               float* partials, int64_t partial_tiles, sldm_stream_t stream);
int     sldm_gru_projected_supported(int32_t I, int32_t H);
int     sldm_gru_input_project_forward(const float* x, int64_t N, int32_t T, int32_t I, int32_t H,
                                       const float* W_ih, const float* b_ih, float* gi, sldm_stream_t stream);
int     sldm_gru_input_wgrad(const float* dgi, const float* x, int64_t N, int32_t T, int32_t I, int32_t H,
                             float* partials, int64_t partial_tiles, sldm_stream_t stream);

/* ---- whole block, host buffers in / host buffers out -----------------------
 * For hosts that own no device memory (the reference-side stub in
 * INTEGRATION.md).  All pointers are HOST pointers.  Parameters of layer l are
 * params_h[5*l + {0:W_l, 1:b_l, 2:W_r, 3:ln_w, 4:ln_b}].  hdims has L+1 entries.
 * Copies inputs to the current device, builds the CSR, runs L layers, copies
 * the result back and synchronises the stream before returning.
 *   forward_host : out_h [N, hdims[L]]
 *   train_host   : additionally takes dout_h [N, hdims[L]] and returns
 *                  dx_h [N, hdims[0]] (may be NULL) and grads_h[5*l+k] laid out
 *                  like params_h.
 */
int sldm_sage_block_forward_host(const float* x_h, const int64_t* edge_index_h,
                                 int64_t N, int64_t E,
                                 const int32_t* hdims, int32_t L,
                                 const float* const* params_h,
                                 float eps, float slope,
                                 float* out_h);
int sldm_sage_block_train_host(const float* x_h, const int64_t* edge_index_h,
                               int64_t N, int64_t E,
                               const int32_t* hdims, int32_t L,
                               const float* const* params_h,
                               float eps, float slope,
                               const float* dout_h,
                               float* out_h, float* dx_h, float* const* grads_h);

#ifdef __cplusplus
}
#endif
#endif /* SLDM_SAGE_H_ */
