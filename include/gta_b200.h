/*
 * gta_b200.h -- C ABI of the B200-native execution backend for the GTA message-passing ISA.
 *
 * The reference (Jagnate/GTA_graph_tensor_acclelrator_for_general_GNN) has NO FFI and no
 * functional execution: its interpreter emits instruction descriptors
 * (vTCAD/code/interpreter.py:132-163, 215-298, 313-479) that only the cycle model
 * (vTCAD/code/simulator.py:281-355 calculate_running_cycle) consumes.  Each entry point
 * below is therefore cited against the ISA instruction / reference function whose work it
 * performs; the Python host (executor.py) binds them with ctypes exactly as
 * INTEGRATION.md shows.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name starts with h_;
 *   - every function returns 0 (GTA_OK) or a GTA_ERR_* code and never throws;
 *     gta_last_error() returns a thread-local message for the last failure;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and nothing
 *     synchronises unless stated;
 *   - the caller owns every buffer; the library allocates nothing persistent;
 *   - feature tables are row-major with an explicit leading dimension `ld*` in ELEMENTS;
 *     rows must be 16-byte aligned (ld % 4 == 0 for fp32) so 128-bit loads are legal;
 *   - adjacency A[row = dst i, col = src j]; CSR rows are destinations, columns ascending
 *     sources (template/ISA_defination.yaml:35; tile walk simulator.py:262-263,292).
 */
#ifndef GTA_B200_H
#define GTA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GTA_OK 0
#define GTA_ERR_INVALID 1      /* bad argument (null pointer, misaligned ld, unsupported width) */
#define GTA_ERR_CUDA 2         /* a CUDA call failed; see gta_last_error() */
#define GTA_ERR_UNSUPPORTED 3  /* legal ISA but no kernel yet */
#define GTA_ERR_WORKSPACE 4    /* workspace too small */

/* epilogue applied while the aggregated row is still in registers (COMP_SF applynode,
 * genGraphOP.py:62 GAT op 13; fused per hardware_info.yaml Inst_fused) */
#define GTA_EPI_NONE 0
#define GTA_EPI_ELU 1
#define GTA_EPI_RELU 2

/* which part of an aggregation call runs.  RESET clears the chain flags of multi-item rows and must run
 * once before the first MAIN launch of a pass; MAIN launches the item kernel over the items handed in.
 * Callers that start a column block as soon as its part of the source table has landed launch
 * RESET|MAIN for the first block's items and MAIN alone for the rest (see h_block_begin). */
#define GTA_PHASE_MAIN 1
#define GTA_PHASE_RESET 2
#define GTA_PHASE_ALL 3
/* hint, OR-ed in: the work list is long and its items are tiny (a low-degree graph): the persistent launch
 * walks it with static striding instead of taking items from a counter (RMAT-20, 16 edges per item: 2.2 ms
 * static against 7.4 ms with batched grabs; the Reddit shape, 160 edges per item, is 20 % faster dynamic) */
#define GTA_PHASE_STATIC 4

/* how the per-edge weight of gta_aggregate_f32 is formed */
#define GTA_W_NONE 0       /* plain sum                       (gather ADD, no applyedge)      */
#define GTA_W_EDGE 1       /* w[k,h]                          (applyedge MUL, GCN op 1 / GAT 11) */
#define GTA_W_EDGE_DIV 2   /* w[k,h] / rowden[i,h]            (GAT op 9 '/', encoded COMP_MUL)  */

const char* gta_last_error(void);
int gta_abi_version(void);
/* number of kernel launches issued by this library since the last reset (for "gpu_launches") */
int64_t gta_launch_count(void);
void gta_launch_count_reset(void);

/* ---------------------------------------------------------------------------------------
 * Graph preprocessing on device.  Replaces the dense-N^2 host path of
 * code/preprocessing.py:12-72 (calculate_sparsity, cal_min_sparsity) and supplies the
 * CSR / partition / reorder steps the north star asks for (no reference implementation;
 * bit-exact against oracle/gta_oracle.py).
 * ------------------------------------------------------------------------------------ */

/* COO -> CSR by (dst, src) ascending, stable.  indptr[N+1] int64, indices[E] int32,
 * perm[E] int64 (may be NULL): perm[k] = input position of CSR edge k.  Duplicate edges are kept (a
 * multigraph).  Synchronises the stream once: an edge whose destination is outside [0, N) or whose source
 * is negative makes the call return GTA_ERR_INVALID (the outputs are then undefined). */
size_t gta_csr_build_workspace(int64_t num_edges, int64_t num_nodes);
int gta_csr_build(const int32_t* dst, const int32_t* src, int64_t num_edges, int64_t num_nodes,
                  int64_t* indptr, int32_t* indices, int64_t* perm,
                  void* workspace, size_t workspace_bytes, void* stream);

/* calculate_sparsity(row = tile_rows, col = 1) (code/preprocessing.py:12-40): counts[tr*N + c]
 * = number of edges with dst in row tile tr and src == c, self loops excluded.  Precondition: no
 * duplicate (dst, src) pairs -- the reference counts non-zeros of a dense adjacency
 * (np.count_nonzero, preprocessing.py:37), where a repeated pair is one entry; a multigraph would be
 * counted per edge here.  graph.calculate_sparsity checks it.
 * Only row tiles [tile_begin, tile_end) are produced (counts has (tile_end-tile_begin)*N
 * entries), so Reddit-size tables can be streamed. */
int gta_tile_nnz(const int64_t* indptr, const int32_t* indices, int64_t num_nodes,
                 int64_t tile_rows, int64_t tile_begin, int64_t tile_end,
                 int32_t* counts, void* stream);
/* cal_min_sparsity (code/preprocessing.py:53-63): maximum entry of the whole table, computed
 * in batches of row tiles inside `workspace` (>= num_nodes*4 bytes; more = fewer passes).
 * *h_max is written on the HOST after an internal stream synchronise. */
int gta_tile_nnz_max(const int64_t* indptr, const int32_t* indices, int64_t num_nodes,
                     int64_t tile_rows, void* workspace, size_t workspace_bytes,
                     int32_t* h_max, void* stream);

/* Destination-range partition balanced by edges: bounds[k] = min r : indptr[r] >= floor(k*E/P). */
int gta_partition(const int64_t* indptr, int64_t num_nodes, int32_t parts, int64_t* bounds,
                  void* stream);

/* Destination-partitioned execution.  The gathered source table of rank r is [parts, stride, F] (each
 * rank's rows padded to `stride`); slot k holds the rows of rank (r + k) mod parts -- `rotate` = r puts the
 * rank's own rows first, rotate = 0 is the layout of a plain all-gather.
 * out[k] = ((p - rotate) mod parts)*stride + (indices[k] - bounds[p]), p = owner of indices[k]. */
int gta_remap_sources(const int32_t* indices, int64_t num_edges, const int64_t* bounds,
                      int32_t parts, int64_t stride, int32_t rotate, int32_t* out, void* stream);

/* ---------------------------------------------------------------------------------------
 * Exchange of the source-side tables INSIDE the aggregation launch (ipc.cu, exchange.cuh, aggregate.cu, gat_aggregate.cu); replaces the
 * per-layer NCCL all-gather of a destination-partitioned run (SURVEY.md section 8e).
 *
 * Every rank owns, per step parity, one gathered table [parts, stride, ld] (gta_ipc_alloc, published to
 * the peers through CUDA IPC) and one signal block (gta_exchange_signal_bytes()).  A step on rank r:
 *   1. the producer (gta_gemm_f32) writes the rank's rows [Z | er] into slot 0 of its table;
 *   2. gta_er_stats over those rows, then gta_exchange_publish: the er range and the step number go to
 *      every peer's signal block (release, system scope);
 *   3. gta_aggregate_f32 / gta_gat_aggregate_f32 with a gta_exchange_t: the first `copy_ctas` CTAs of the
 *      launch pull slot 0 of peer (r + k) mod parts over NVLink into slot k of the local table, k = 1 ..
 *      parts-1 in ring order, waiting for that peer's step number first; the other CTAs walk the work list
 *      (column blocks = the own slot, then groups of peer slots in ring order) and wait, per item, until the
 *      slot of the item's last source has landed (slots land in order).
 * No collective library call, no SMs taken by a communication kernel, no launch boundary between transfer
 * and compute.  Tables are double-buffered by step parity: a peer is at most one step ahead.
 * Every wait is bounded (a rank that never publishes makes the others trap, it does not hang the GPU).
 * ------------------------------------------------------------------------------------ */
#define GTA_MAX_RANKS 16
typedef struct {
  int32_t world;                        /* parts; <= GTA_MAX_RANKS */
  int32_t rank;
  int32_t step;                         /* >= 1, the same on every rank, +1 per layer execution */
  int32_t copy_ctas;                    /* CTAs that pull (0: library default) */
  int64_t slot_rows;                    /* stride: rows per slot = col_block of the work list */
  int64_t row_bytes;                    /* bytes per table row (ld * 4), multiple of 16 */
  void* table;                          /* this rank's table for this step */
  void* signals;                        /* this rank's signal block */
  const void* peer_table[GTA_MAX_RANKS];/* [k]: table (this step's parity) of rank (rank + k) mod world */
  int64_t slot_valid_rows[GTA_MAX_RANKS];/* [k]: rows of rank (rank + k) mod world */
} gta_exchange_t;
size_t gta_exchange_signal_bytes(void);
/* `stats` = this rank's er range as gta_er_stats(er, lder, rows, 0, heads, stats) wrote it (2*heads uint32;
 * NULL with heads = 0: none, the consumers run the online softmax -- GCN, or a head count gta_er_stats
 * refuses).  h_peer_signals[q] is the signal block of rank q as mapped in this process ([rank] = its own). */
int gta_exchange_publish(const uint32_t* stats, int32_t heads, int32_t rank, int32_t world, int32_t step,
                         void* const* h_peer_signals, void* stream);

/* Peer-to-peer plumbing: buffers that can be mapped by the other ranks of the box.  gta_ipc_alloc'ed
 * buffers are the only memory this library owns; free them with gta_ipc_free.  handle64 is a 64-byte
 * cudaIpcMemHandle_t. */
int gta_ipc_alloc(size_t bytes, void** ptr);
int gta_ipc_free(void* ptr);
int gta_ipc_export(void* ptr, uint8_t* handle64);
int gta_ipc_open(const uint8_t* handle64, void** mapped);
int gta_ipc_close(void* mapped);

/* Degree reorder: perm[new] = old, descending in-degree, stable. */
size_t gta_reorder_workspace(int64_t num_nodes);
int gta_reorder(const int64_t* indptr, int64_t num_nodes, int64_t* perm,
                void* workspace, size_t workspace_bytes, void* stream);

/* Work list for the aggregation kernels (schedule.cu).  Rows [row_begin,row_end) are cut into
 * ITEMS: at most `chunk` consecutive CSR edges of one destination row whose sources all fall in
 * one column block of `col_block` source ids (col_block <= 0 or >= num_sources: no blocking).
 * Items are ordered by (column block, row, position) so the CTAs resident at any moment gather
 * from one L2-sized slice of the source table; this is the B200 form of the reference's
 * TR x TC tile walk (interpreter.py:85-106; simulator.py:262-263,292).
 *   items     int32[4] per item = {row - row_begin, edge_begin, edge_count, partial slot | -1}
 *   row_slots int32[rows+1]: slots of row r are [row_slots[r], row_slots[r+1]) (empty if 1 item);
 *             the items of a row carry consecutive slots in work-list order (the fold order)
 * h_counts[0] = number of items, h_counts[1] = number of partial slots; h_block_begin[cb] = first
 * item of column block cb, h_block_begin[n_cb] = number of items (host arrays, after a sync;
 * n_cb = gta_schedule_col_blocks(num_sources, col_block)). */
int32_t gta_schedule_col_blocks(int64_t num_sources, int64_t col_block);
size_t gta_schedule_workspace(int64_t num_rows, int64_t num_sources, int64_t col_block);
int64_t gta_schedule_max_items(int64_t num_rows, int64_t num_edges, int32_t chunk,
                               int64_t num_sources, int64_t col_block);
int gta_schedule_build(const int64_t* indptr, const int32_t* indices, int64_t row_begin,
                       int64_t row_end, int64_t num_sources, int32_t chunk, int64_t col_block,
                       int32_t* items, int64_t items_capacity, int32_t* row_slots,
                       int64_t* h_counts, int64_t* h_block_begin, void* workspace,
                       size_t workspace_bytes, void* stream);
/* The same with explicit column blocks: block b holds the sources in [h_cuts[b-1], h_cuts[b]) (h_cuts[-1] = 0,
 * the last block everything from h_cuts[num_cuts-1] on); num_cuts + 1 blocks, host array of ascending positive
 * source ids.  An exchange uses it to walk its own slot, then a few GROUPS of peer slots (dist.py): per-slot
 * blocks cut an 8-GPU Reddit-shape row into 8 items of 61 edges and lost 47 % to per-item overhead.
 * Workspace / capacity: gta_schedule_workspace(rows, num_cuts + 1, 1), gta_schedule_max_items(rows, E, chunk,
 * num_cuts + 1, 1). */
int gta_schedule_build_cuts(const int64_t* indptr, const int32_t* indices, int64_t row_begin,
                            int64_t row_end, int32_t chunk, const int64_t* h_cuts, int32_t num_cuts,
                            int32_t* items, int64_t items_capacity, int32_t* row_slots,
                            int64_t* h_counts, int64_t* h_block_begin, void* workspace,
                            size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * COMP_MM (applynode)  --  interpreter.py:145-161 with Weight_Size; simulator.py:338-341.
 * Z[N,F] = X[N,K] . W[K,F]  (template/ISA_defination.yaml:28-31, einsum j,ij->i).
 * Optional fused GAT ops 1,2 (genGraphOP.py:50-51): el = Z.Al, er = Z.Ar with Al,Ar [F,H]
 * row-major dense; pass NULL to skip.  el is dense [N,H]; er has row stride `lder` elements
 * (0 = dense), so a partitioned run can write z and er straight into its slot of the gathered
 * [F | H] source table.  fp32 in / fp32 out.  Error bound, with s = sum_k |x_k w_k|:
 * FFMA path |z - z64| <= 1e-5 |z64| + 1e-5 s.  tcgen05 path: the same plus 2^-26 K s, because
 * its fp32 accumulator loses about 1.2e-8 K relative on same-sign data (measured on an NVIDIA
 * B200 at 1000 W: 7.8e-6 at K = 602, 1.7e-5 at K = 1433, 4.7e-5 at K = 4096; FFMA 1.5e-6,
 * 2.3e-6, 3.8e-6).  With terms of mixed sign the error cancels and both paths hold 1e-5.
 * ------------------------------------------------------------------------------------ */
/* `workspace` (gta_gemm_workspace(k,f) bytes, 128-byte aligned) holds the hi/lo TF32 split of W
 * for the tensor-core kernel; without it the call takes the FFMA kernel. */
size_t gta_gemm_workspace(int32_t k, int32_t f);
int gta_gemm_f32(const float* x, int64_t ldx, const float* w, int64_t ldw,
                 float* z, int64_t ldz, int64_t num_rows, int32_t k, int32_t f,
                 const float* al, const float* ar, int32_t heads, float* el, float* er,
                 int64_t lder, void* workspace, size_t workspace_bytes, void* stream);
/* bf16 STORAGE MODE (SURVEY.md section 8d; the reference's IR declares data_format FP16,
 * template/IR_defination.yaml:10-27): the gathered table Z is stored in bf16, everything is accumulated in
 * fp32.  Tolerance of the mode: rtol 2e-2, atol 1e-2 * rowscale.  gta_gemm_f32_zbf16 is gta_gemm_f32 with Z
 * rounded to bf16 once, in the epilogue (z: bf16 rows, ldz in bf16 elements, a multiple of 8; el / er fp32 from
 * the fp32 accumulators; tcgen05 kernel only).  gta_aggregate_bf16 / gta_gat_aggregate_bf16 are the
 * aggregation entry points over such a table (x / z: bf16 rows, ldx / ldz in bf16 elements, f a multiple of
 * 8, per-head width a multiple of 8; out, partials, weights, el, er stay fp32; head counts 1, 2, 4). */
int gta_gemm_f32_zbf16(const float* x, int64_t ldx, const float* w, int64_t ldw,
                       void* z, int64_t ldz, int64_t num_rows, int32_t k, int32_t f,
                       const float* al, const float* ar, int32_t heads, float* el, float* er,
                       int64_t lder, void* workspace, size_t workspace_bytes, void* stream);
int gta_aggregate_bf16(const int32_t* items, int64_t num_items, const int32_t* row_slots,
                       int64_t num_slots, const int32_t* indices,
                       int32_t wmode, const float* w, int32_t wh, const float* rowden,
                       const void* x, int64_t ldx, float* out, int64_t ldo, int32_t f,
                       int32_t epilogue, float* partials, int32_t* chain_state,
                       const gta_exchange_t* exchange, int32_t phases, void* stream);
int gta_gat_aggregate_bf16(const int32_t* items, int64_t num_items, const int32_t* row_slots,
                           int64_t num_slots, const int32_t* indices,
                           const float* el, const float* er, int64_t lder, int32_t heads, float slope,
                           const void* z, int64_t ldz, float* out, int64_t ldo, int32_t f,
                           int32_t epilogue, float* rowmax, float* rowsum,
                           float* partials, int32_t* chain_state, const uint32_t* er_stats,
                           int64_t col_block, const gta_exchange_t* exchange, int32_t phases,
                           void* stream);

/* kernel choice of gta_gemm_f32: 0 = auto (tcgen05 3xTF32 when the shape is eligible, else
 * FFMA), 1 = force the FFMA kernel, 2 = force tcgen05 (GTA_ERR_UNSUPPORTED if ineligible). */
int gta_gemm_set_mode(int mode);
int gta_gemm_get_mode(void);

/* ---------------------------------------------------------------------------------------
 * COMP_MUL_COMP_ADD (fused applyedge MUL + gather ADD R; hardware_info.yaml:35-38,
 * interpreter.py:575-638) and plain COMP_ADD gather (interpreter.py:85-106):
 *   out[i,:] = epi( sum_{k in row i, ascending src} weight(k) (x) x[src(k),:] )
 * `w` is [E,wh] (wh = 1 scalar per edge, or wh = heads, head h covering f/wh features);
 * `rowden` is [N,wh] for GTA_W_EDGE_DIV.  Work comes from gta_schedule_build; the launch is persistent
 * (warps take items from a counter in work-list order).  Rows that own several items are folded in slot
 * order INSIDE the kernel (each item waits for its predecessor's state, no merge launch): `partials`
 * holds num_slots*f floats (NULL when num_slots == 0); `chain_state` holds, for W = ceil(f/128) feature
 * windows, W*num_slots int32 chain flags (cleared by GTA_PHASE_RESET) followed by W + GTA_MAX_RANKS int32
 * (item counters and slot-arrival counters, cleared by every MAIN launch) and is always required.
 * `exchange` (NULL: the source table is complete) makes the launch pull the peers' slots itself, see
 * gta_exchange_t; the work list's column blocks must then end on slot boundaries (multiples of
 * exchange->slot_rows), the first block being slot 0 alone.
 * ------------------------------------------------------------------------------------ */
int gta_aggregate_f32(const int32_t* items, int64_t num_items, const int32_t* row_slots,
                      int64_t num_slots, const int32_t* indices,
                      int32_t wmode, const float* w, int32_t wh, const float* rowden,
                      const float* x, int64_t ldx, float* out, int64_t ldo, int32_t f,
                      int32_t epilogue, float* partials, int32_t* chain_state,
                      const gta_exchange_t* exchange, int32_t phases, void* stream);

/* Edge phase "sum of up to three terms, a unary, the row sum" in one pass -- PNA ops 5-8
 * (vTCAD/GraphOP/genGraphOP.py:110-147: gather_R(SF(edge + scatterC(a) + scatterR(b)))):
 *     out[i, :] = epilogue( sum_{k in row i} unary( edge[k, :] + x[src_k, :] + rowterm[i, :] ) )
 * edge [E, lde] in CSR edge order, x [num_sources, ldx] gathered by source, rowterm [N, ldr]; any of the three
 * may be NULL (not all).  unary: GTA_UN_* (GTA_UN_COPY = identity; slope for GTA_UN_EXP_LEAKY_RELU).  fp32,
 * f % 4 == 0, 16-byte aligned rows.  Same work list, chain state and phases as gta_aggregate_f32 (partials:
 * num_slots * f floats); ascending-edge reduction, bitwise reproducible.  Nothing E x F is written. */
int gta_aggregate_edge_sum_f32(const int32_t* items, int64_t num_items, const int32_t* row_slots,
                               int64_t num_slots, const int32_t* indices,
                               const float* edge, int64_t lde, const float* x, int64_t ldx,
                               const float* rowterm, int64_t ldr, int32_t unary, float slope,
                               float* out, int64_t ldo, int32_t f, int32_t epilogue,
                               float* partials, int32_t* chain_state, int32_t phases, void* stream);

/* Measured ceiling of the gather kernels (roofline denominator, not part of the path): every resident
 * lane group gathers `gathers_per_group` pseudo-random rows of `table` ([rows, ld] fp32, f <= 128 features
 * read per row) with the aggregation kernels' own load instruction and nothing else.  Returns the number of
 * groups that ran (> 0) or a negative error code (-GTA_ERR_*); time it with events around the call.
 * `sink` needs 16 bytes per group (never written in practice). */
int gta_gather_peak_probe(const float* table, int64_t rows, int64_t ld, int32_t f, int64_t gathers_per_group,
                          float* sink, void* stream);

/* Range of the GAT source-side logits per column block: stats[cb][0][h] / stats[cb][1][h] = ordered-int
 * codes of max_j er[j,h] and max_j -er[j,h] over the sources j of column block cb (col_block source ids
 * per block, <= 0: one block; 2*H uint32 per block).  heads must be a power of two <= 32
 * (GTA_ERR_UNSUPPORTED otherwise).  gta_gat_aggregate_f32 uses it to shift the softmax by the bound
 * leaky_relu(el[i,h] + max er) instead of a running maximum (genGraphOP.py:56-58 ops 6-8). */
int gta_er_stats(const float* er, int64_t lder, int64_t num_sources, int64_t col_block, int32_t heads,
                 uint32_t* stats, void* stream);

/* ---------------------------------------------------------------------------------------
 * GAT edge phase in ONE pass (ops 3-13 of genGraphOP.py:52-62; ISA blocks
 * [4,5,6,7,8] + [3,9,10,11,12,13] of SURVEY Appendix B3 collapsed):
 *   s = el[i,h] + er[j,h]; e = leaky_relu(s, slope); alpha = softmax_row(e);
 *   out[i,:] = epi( sum_k alpha[k,h(f)] * z[j,:] )
 * el [rows,H] (dense) is indexed by LOCAL row; er (row stride `lder` elements, so it can live in
 * the same gathered table as z: [.., F | H] per source) and z by source id.
 * partials: num_slots * gta_gat_partial_stride(f,H) floats (acc[f], then (max[H], sum[H]) padded to 4
 * per 128-feature window); chain_state as for gta_aggregate_f32.
 * er_stats (from gta_er_stats with the same col_block; NULL: online softmax with a running maximum):
 * where a block's er range is below 60 the softmax is shifted by a per-(row, block) bound -- same result
 * within rounding, no warp reductions.  With `exchange` the statistics are taken from the signal block
 * (published by the slot owners) and er_stats / col_block are ignored.  Optionally emits rowmax[N,H] and
 * rowsum[N,H] (NULL to skip; asking for rowmax selects the online path, which tracks the true maximum).
 * ------------------------------------------------------------------------------------ */
int32_t gta_gat_partial_stride(int32_t f, int32_t heads);
int gta_gat_aggregate_f32(const int32_t* items, int64_t num_items, const int32_t* row_slots,
                          int64_t num_slots, const int32_t* indices,
                          const float* el, const float* er, int64_t lder, int32_t heads, float slope,
                          const float* z, int64_t ldz, float* out, int64_t ldo, int32_t f,
                          int32_t epilogue, float* rowmax, float* rowsum,
                          float* partials, int32_t* chain_state, const uint32_t* er_stats,
                          int64_t col_block, const gta_exchange_t* exchange, int32_t phases,
                          void* stream);

/* GAT block [4,5,6,7,8] alone (COMP_ADD 6, COMP_SF 7, STORE_E 7, COMP_ADD 8 gather):
 *   p[k,h] = exp(leaky_relu(el[i,h] + er[j,h]) - rowmax[i,h]),  rowsum[i,h] = sum_k p[k,h].
 * One warp per row (no chunking); p is [E,H] in CSR edge order. */
int gta_gat_logits_f32(const int64_t* indptr, const int32_t* indices, int64_t row_begin,
                       int64_t row_end, const float* el, const float* er, int32_t heads,
                       float slope, int32_t stabilize, float* p, float* rowmax, float* rowsum,
                       void* stream);

/* ---------------------------------------------------------------------------------------
 * Generic single-op kernels so that ANY legal plan executes (SURVEY section 8f-1).
 * Edge operands are either materialised [E,width] tensors or VIRTUAL scatters
 * (FETCH eliminated by fuse_fetch, interpreter.py:768-806): kind 0 = edge tensor,
 * 1 = node tensor indexed by dst (scatter R), 2 = node tensor indexed by src (scatter C).
 * ------------------------------------------------------------------------------------ */
#define GTA_OPND_EDGE 0
#define GTA_OPND_DST 1
#define GTA_OPND_SRC 2
#define GTA_BIN_ADD 0
#define GTA_BIN_MUL 1
#define GTA_BIN_DIV 2       /* a / b, and 0 where b == 0 (rows without edges) */
#define GTA_UN_EXP_LEAKY_RELU 0
#define GTA_UN_ELU 1
#define GTA_UN_RELU 2
#define GTA_UN_COPY 3

/* out[k,:] = a[k,:] (op) b[k,:] over edges of rows [row_begin,row_end); widths wa, wb divide wo
 * (head broadcast).  COMP_ADD / COMP_MUL applyedge. */
int gta_edge_binary_f32(const int64_t* indptr, const int32_t* indices, int64_t row_begin,
                        int64_t row_end, int32_t op,
                        const float* a, int32_t kind_a, int32_t wa, int64_t lda,
                        const float* b, int32_t kind_b, int32_t wb, int64_t ldb,
                        float* out, int32_t wo, int64_t ldo, void* stream);
/* out[k,:] = f(a[k,:]); COMP_SF applyedge (exp(leaky_relu)) or a materialising scatter (COPY). */
int gta_edge_unary_f32(const int64_t* indptr, const int32_t* indices, int64_t row_begin,
                       int64_t row_end, int32_t op, float slope,
                       const float* a, int32_t kind_a, int32_t wa, int64_t lda,
                       float* out, int64_t ldo, void* stream);
/* node elementwise: out = a (op) b  /  out = f(a)  (COMP_ADD/MUL/SF applynode) */
int gta_node_binary_f32(int32_t op, const float* a, int32_t wa, int64_t lda,
                        const float* b, int32_t wb, int64_t ldb,
                        float* out, int32_t wo, int64_t ldo, int64_t num_rows, void* stream);
int gta_node_unary_f32(int32_t op, float slope, const float* a, int64_t lda, float* out,
                       int64_t ldo, int32_t width, int64_t num_rows, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GTA_B200_H */
