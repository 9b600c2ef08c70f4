/*
 * kgc_b200.h - C ABI of libkgc_b200.so, the B200 (sm_100a) implementation of the M-GCN
 * hot path (weilonghu/KGC-GCN).  The reference is pure Python and has no FFI of its own;
 * each entry point below names the reference code (file:line under the reference root) whose
 * arithmetic it replaces.  The Python host layer (kgc_gcn_b200/*.py) binds these with ctypes
 * and keeps the reference's module API (MGCN / MGCNConv / ConvE / DataLoader); INTEGRATION.md
 * shows the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - extern "C"; every function returns int: 0 = OK, non-zero = failure, text in
 *     kgc_last_error() (thread-local).  No torch types, plain device pointers and sizes.
 *   - The CALLER allocates every input, output and workspace buffer (device memory) and
 *     passes the CUDA stream (a cudaStream_t cast to void*); nothing is synchronised
 *     internally except where a function says so; no hidden global state.
 *   - Matrices are row-major and dense unless a stride is given.  D (= gcn_in_dim) must be
 *     a multiple of 4 and <= 256; Dout a multiple of 4 and <= 1024 (float4 paths).
 *   - Index dtypes: the reference's int64 edge lists are consumed as they are by
 *     kgc_csr_build; everything downstream is int32 (node, edge and type ids < 2^31).
 *   - There is NO CPU fallback: every entry point launches sm_100a kernels.
 */
#ifndef KGC_B200_H_
#define KGC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define KGC_ABI_VERSION 4

/* Work item of a fix-up reduction level: rows [beg, end) of the carry / partial array are summed;
 * the result goes to row `out` of the final output (flags & 1) or of the partial buffer of this
 * level (flags & 1 == 0); flags >> 1 = the final row.  Built by the host plan (kgc_gcn_b200/plan.py). */
typedef struct { int32_t beg, end, out, flags; } kgc_item_t;

/* Streaming aggregation (K2/K3): the sorted records are cut into chunks of KGC_CHUNK_EDGES; a chunk's
 * leading row that began in an earlier chunk goes to carry row head_slot when it ends inside the chunk, the
 * row still open at the end of the chunk goes to carry row tail_slot (-1 = not needed).  rowflags[p] of a
 * sorted record = output row | first-record-of-its-row << 30 | last-record-of-its-row << 31. */
#define KGC_CHUNK_EDGES 32
typedef struct { int32_t head_slot, tail_slot; } kgc_chunk_t;

/* Edge record of a sorted CSR: 16 bytes, one 128-bit load per edge.
 *   dst-sorted : a = src,  b = type      src-sorted : a = dst, b = type
 *   type-sorted: a = src,  b = dst       eid is the GLOBAL edge id (0..2E-1); norm is fp32 */
typedef struct { int32_t eid, a, b; float norm; } kgc_edge_rec_t;

const char* kgc_last_error(void);
int kgc_abi_version(void);

/* ---- K1: CSR / permutation builder + per-half degree normalisation -------------------------
 * Replaces MGCNConv.compute_norm (model.py:72-80) and the gather/scatter index handling of PyG
 * propagate (model.py:99-101).  Input is the reference's edge list: src = edge_index[0],
 * dst = edge_index[1], type = edge_attr[0], all int64 [n_edges2]; the first n_edges2/2 edges
 * are the "in" half, the rest the "out" half (model.py:84-90).
 *   deg[h*N + v]  = #{e in half h : src_e = v}                       (int32, exact)
 *   norm[e]       = deg_h^-1/2[src_e] * deg_h^-1/2[dst_e], 0 where a degree is 0   (fp32)
 *   perm_K / rowptr_K / rec_K for K in {dst, src, type}: STABLE sort of all n_edges2 edges by
 *   key K (ties keep ascending edge id, so within a row the in-half edges come first);
 *   rowptr_K[r] = first sorted position with key >= r; rowmid_dst[r] = first position in
 *   row r whose edge belongs to the out half.
 * Synchronises the stream once (to validate ids); ids out of range are an error. */
size_t kgc_csr_workspace_bytes(int64_t n_edges2, int64_t n_nodes, int64_t n_types);
/* Partitioned graphs (SURVEY.md 8(e): nodes range-partitioned by destination): a rank passes only the
 * edges it owns, in-half edges first (n_edges_in of them), src as GLOBAL node ids in [0, n_nodes), dst
 * as LOCAL row ids in [0, n_dst_rows) with global id = dst + dst_offset, and the GLOBAL per-half degrees
 * (deg_given = 1; deg is then an input).  The single-GPU case is n_edges_in = n_edges2 / 2,
 * n_dst_rows = n_nodes, dst_offset = 0, deg_given = 0. */
int kgc_csr_build(const int64_t* src, const int64_t* dst, const int64_t* type,
                  int64_t n_edges2, int64_t n_edges_in, int64_t n_nodes, int64_t n_dst_rows, int64_t dst_offset,
                  int64_t n_types, int32_t deg_given, int32_t* deg, float* norm,
                  int32_t* perm_dst, int32_t* rowptr_dst, int32_t* rowmid_dst, kgc_edge_rec_t* rec_dst,
                  int32_t* perm_src, int32_t* rowptr_src, kgc_edge_rec_t* rec_src,
                  int32_t* perm_type, int32_t* rowptr_type, kgc_edge_rec_t* rec_type,
                  int64_t type_block_rows, void* workspace, size_t workspace_bytes, void* stream);
/* type_block_rows > 0: the type sort is BLOCKED BY SUBJECT ROW.  Its key becomes (s / type_block_rows) * n_types + type,
 * s = the edge's subject (src of an in-half edge, dst of its reverse): kgc_csr_type_rows(...) = ceil(n_nodes /
 * type_block_rows) * n_types key rows (rowptr_type has that many + 1 entries; pass it as n_types to
 * kgc_csr_workspace_bytes).  The d_rel pass (kgc_agg_bwd_rel) gathers x[src] and g[dst] at random; with the blocked order
 * the rows a block touches (2 * type_block_rows * 4 D bytes + the hub objects) stay in the 126 MB L2 and are read from
 * HBM once - at the Wikidata5M shape that pass moved 42 GB for 16.5 GB of edge rows.  The pass then yields one partial
 * row per (block, type); kgc_block_sum adds the blocks in ascending order (deterministic). */
int64_t kgc_csr_type_rows(int64_t n_nodes, int64_t n_types, int64_t type_block_rows);
/* out[i] = sum over b < n_blocks (ascending) of in[b * n + i], i < n (n a multiple of 4). */
int kgc_block_sum(const float* in, int64_t n_blocks, int64_t n, float* out, void* stream);

/* Streaming schedules of K2/K3 on the device.  The sorted records of an aggregation are cut into chunks of `chunk` (32)
 * records, one warp each; segments [seg_beg[s], seg_end[s]) tile the record array in order (empty segments allowed) and
 * reduce into output row seg_row[s].  Writes rowflags[p] = row | first-record-of-its-segment << 30 | last << 31,
 * rec_seg[p] = the segment of record p (scratch), and per chunk c inter[2c] / inter[2c + 1] = 1 when the chunk needs a
 * head / tail carry row (its first segment began in an earlier chunk and ends here / its last segment continues).
 * Slot numbers = exclusive prefix sum of inter.  Bit-exact against plan.build_stream_plan (numpy). */
int kgc_stream_plan_flags(const int32_t* seg_beg, const int32_t* seg_end, const int32_t* seg_row, int64_t n_seg,
                          int64_t n_rec, int32_t chunk, uint32_t* rowflags, int32_t* rec_seg, int32_t* inter, void* stream);

/* ---- K2: aggregation forward -----------------------------------------------------------------
 * Replaces the gather + MGCNConv.message product + norm + scatter-add of the "in" and "out"
 * propagations (model.py:99-100,111-118) in the aggregate-then-transform order:
 *   out[row] = sum over the row's records of  norm_e * x[a_e] (.) rel[b_e] (.) ee[eid_e]
 * over dst-sorted records (row = plane * n_dst_rows + dst; plane 0 = in half, 1 = out half);
 * deterministic (fixed order, no float atomics).  Rows that lie inside one chunk are written to
 * out_final, chunk-boundary rows to carry (reduced by kgc_rows_reduce), rows without records by
 * kgc_rows_fill.  x [n_nodes,D], rel [n_types,D], ee [n_edges2,D], out_final [*,D], carry [*,D]. */
int kgc_agg_fwd(const float* x, const float* rel, int64_t n_types, const float* ee,
                const kgc_edge_rec_t* rec_dst, const uint32_t* rowflags, const kgc_chunk_t* chunks, int64_t n_rec,
                float* out_final, float* carry, int32_t D, void* stream);

/* out[rows[i]] = addend ? addend[rows[i]] : 0 for the rows no record maps to. */
int kgc_rows_fill(const int32_t* rows, int64_t n_rows, const float* addend, float* out, int32_t D, void* stream);

/* Fix-up levels shared by K2/K3: out[row] = sum of rows [beg,end) of `part_in` (carry rows, then partial
 * rows of the previous level) (+ addend[row] on final rows when addend != NULL), in a fixed order.  The first
 * n_large items get a 512-thread block each (hub rows), the others one 8-lane group each. */
int kgc_rows_reduce(const float* part_in, const kgc_item_t* items, int64_t n_items, int64_t n_large,
                    float* out_final, float* out_part, const float* addend, int32_t D, void* stream);

/* ---- K3: aggregation backward ------------------------------------------------------------------
 * Autograd of the same three lines (model.py:114-118 + aggr='add').  g3 is [2,n_dst_rows,D]:
 * plane 0/1 = d(agg_in)/d(agg_out) = d(res_h) @ W_h^T, indexed by the (local) destination row.
 * Over src-sorted records (row j = source node, global id):
 *   p_e      = norm_e * g3[half_e][a_e] (.) rel[b_e]
 *   d_ee[e]  = p_e (.) x[j]                                  (one row per edge, no reduction)
 *   d_x[j]   = sum_e p_e (.) ee[e]   (+ loop_addend[j], the self-loop term, on final rows when not NULL)
 * half_e = (eid_e >= n_edges_in). */
int kgc_agg_bwd_src(const float* x, const float* rel, int64_t n_types, const float* ee, const float* g3,
                    const kgc_edge_rec_t* rec_src, const uint32_t* rowflags, const kgc_chunk_t* chunks, int64_t n_rec,
                    int64_t n_dst_rows, int64_t n_edges_in, const float* loop_addend,
                    float* d_ee, float* dx_final, float* carry, int32_t D, void* stream);

/* Over type-sorted records (row t = relation type):
 *   d_rel[t] = sum_e norm_e * g3[half_e][b_e] (.) x[a_e] (.) ee[e] */
int kgc_agg_bwd_rel(const float* x, const float* ee, const float* g3,
                    const kgc_edge_rec_t* rec_type, const uint32_t* rowflags, const kgc_chunk_t* chunks, int64_t n_rec,
                    int64_t n_dst_rows, int64_t n_edges_in,
                    float* drel_final, float* carry, int32_t D, void* stream);

/* ---- K3, factorized by (row, type) group (single GPU; kgc_gcn_b200/plan.py GroupedPlan) -------------------------------
 * A knowledge graph's objects are hubs that see each relation type many times, so a sum over edges that carries a factor
 * rel[type] can be regrouped: sum_e rel[t_e] (.) y_e = sum_groups rel[t] (.) (sum over the group's edges of y_e).  The
 * grouped forward stream (kgc_agg_fwd on GroupedPlan records, whose in-half records carry the index of a row of ones)
 * writes P[g] = sum_{e in g} norm_e x[src_e] (.) ee[e] per (dst, type) group of the in half.
 *
 * kgc_agg_bwd_src_grouped: the d_x / d_ee pass over the grouped src-sorted records.  rowflags hold the OUTPUT row of each
 * record: its source row j for an in-half record (as kgc_agg_bwd_src) or n_dst_rows + g for an out-half record of group g
 * (its (src, type) run); xrow[p] = the source row of record p.
 *   d_ee[e]              = norm_e * g3[half_e][a_e] (.) rel[b_e] (.) x[xrow_e]      (bit-identical to kgc_agg_bwd_src)
 *   out[j]               = sum over the in-half records of row j of that product with ee[e] in place of x (+ loop_addend[j])
 *   out[n_dst_rows + g]  = sum_{e in g} norm_e * g3[1][a_e] (.) ee[e]              (Q: no relation factor)
 * loop_addend must have n_dst_rows + n_groups rows whose group rows are zero (the fix-up levels add it on every final row).
 *
 * kgc_group_reduce: first level of a deterministic reduction over groups.  Item k (items[k] = beg, end, out, flags as for
 * kgc_rows_reduce, end - beg <= 32) computes
 *   s = sum over i in [beg, end), ascending, of mult[mrow[i]] (.) part[prow ? prow[i] : i]
 * and writes it to out_final[out] (flags & 1; plus the row's previous value when accumulate != 0) or to out_part[out].
 * Longer segments continue on kgc_rows_reduce levels (addend = out_final itself to accumulate). */
int kgc_agg_bwd_src_grouped(const float* x, const float* rel, int64_t n_types, const float* ee, const float* g3,
                            const kgc_edge_rec_t* rec, const uint32_t* rowflags, const uint32_t* xrow,
                            const kgc_chunk_t* chunks, int64_t n_rec, int64_t n_dst_rows, int64_t n_edges_in,
                            int64_t n_groups, const float* loop_addend, float* d_ee, float* out_final, float* carry,
                            int32_t D, void* stream);
int kgc_group_reduce(const float* part, const int32_t* prow, const float* mult, const int32_t* mrow,
                     const kgc_item_t* items, int64_t n_items, float* out_final, float* out_part, int32_t accumulate,
                     int32_t D, void* stream);

/* ---- K4: layer tail ------------------------------------------------------------------------------
 * Replaces model.py:103-106: out = (drop(in_res) + drop(out_res) + loop_res) / 3 [+ bias];
 * BatchNorm1d over the node rows; tanh.  res3 is [3,n_rows,Dout] (in, out, loop planes).
 * Dropout (nn.Dropout on in_res and out_res, model.py:103): either injected uint8 keep masks mask_in / mask_out
 * [n_rows,Dout] (tests replay the reference's own draws this way), or - masks NULL, seed != NULL, drop_p > 0 - a
 * counter-based Philox4x32-10 stream keyed by *seed (device int64), counter = (float4 index, plane): the forward
 * and the backward regenerate the same mask, nothing is stored.  keep_scale = 1/(1-p).  kgc_dropout_mask writes
 * the mask of one plane (0 = in, 1 = out) for inspection.
 *   kgc_tail_fwd           writes pre[n_rows,Dout] and per-block column partials (sum, sum of squares; fp64) and, when keep
 *                          is given (uint8 [n_rows, kgc_keep_pitch()], Dout <= 256), the keep flags it used: byte c of a
 *                          row = columns 4c..4c+3, low nibble = in half, high nibble = out half.  The backward GEMMs
 *                          apply them to ONE upstream plane while splitting it (the keep argument of kgc_gemm_nt_batch
 *                          and kgc_gemm_tn_tc_batch): no mask is regenerated, no masked plane is written.
 *                          Compacted in / out planes (the layer's sparse halves): slot_h (NULL: plane h is read densely
 *                          from res3) = int32 [n_rows], the row of node row r in rows_h [n_c, Dout], or -1 for a row
 *                          without edges, which contributes exactly 0.  res3's plane h is not read when slot_h is given.
 *                          Same arithmetic order, dropout draws and keep flags.
 *   kgc_colsum_finalize    reduces the partials in a fixed order into sums[2,Dout] (fp64).  A partitioned
 *                          graph all-reduces these 2*Dout doubles across ranks here (SURVEY.md 8(e)).
 *   kgc_colstats_from_sums stats[0]=mean, [1]=biased var, [2]=rstd=1/sqrt(var+eps) over n_rows (GLOBAL) rows
 *                          when training, or from the running statistics (training == 0)
 *   kgc_tail_apply         all_ent = tanh((pre - mean) * rstd * gamma + beta) */
int64_t kgc_tail_num_blocks(int64_t n_rows);
int kgc_dropout_mask(const int64_t* seed, int32_t plane, float drop_p, int64_t n_elem, uint8_t* mask, void* stream);
int32_t kgc_keep_pitch(void);
int kgc_tail_fwd(const float* res3, const int32_t* slot_in, const float* rows_in, const int32_t* slot_out,
                 const float* rows_out, const uint8_t* mask_in, const uint8_t* mask_out, const int64_t* seed,
                 float drop_p, float keep_scale, const float* bias, int64_t n_rows, int32_t Dout, float* pre,
                 double* partials, uint8_t* keep, void* stream);
/* dst[dst_rows[j]] = src[src_rows[j]] for j < n, rows of D floats (D, ld_src, ld_dst multiples of 4); a NULL row list is
 * the identity.  Gathers the occupied rows of a plane into a compact block and scatters them back. */
int kgc_rows_copy(const float* src, int64_t ld_src, const int32_t* src_rows, float* dst, int64_t ld_dst,
                  const int32_t* dst_rows, int64_t n, int32_t D, void* stream);
int kgc_colsum_finalize(const double* partials, int64_t n_blocks, int32_t Dout, double* sums, void* stream);
int kgc_colstats_from_sums(const double* sums, int64_t n_rows, int32_t Dout, float eps, int32_t training,
                           const float* running_mean, const float* running_var, float* stats, void* stream);
/* Single-GPU training (no all-reduce between the two steps): kgc_colsum_finalize + kgc_colstats_from_sums + the
 * running-statistics bookkeeping of nn.BatchNorm1d in ONE launch: running_mean/var (NULL: not tracked) get the momentum
 * update with the unbiased variance, *num_batches_tracked (NULL: skipped) is incremented; sums (NULL: skipped) as above.
 * kgc_colsum_finalize2 = kgc_colsum_finalize plus an fp32 copy of the sums (d_beta / d_gamma of the backward). */
int kgc_colstats_finalize(const double* partials, int64_t n_blocks, int64_t n_rows, int32_t Dout, float eps,
                          float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                          double* sums, float* stats, void* stream);
int kgc_colsum_finalize2(const double* partials, int64_t n_blocks, int32_t Dout, double* sums, float* sums32,
                         void* stream);
/* out_seed != NULL and out_drop_p > 0: dropout of the OUTPUT in the same pass (MGCN.forward's F.dropout(all_ent, gcn_drop),
 * model.py:34): Philox stream of *out_seed, plane 2 (kgc_dropout_mask(seed, 2, p) shows the mask), kept values x 1/(1-p);
 * the keep flags go to out_keep [n_rows, kgc_keep_pitch()] (low nibble of byte c = columns 4c..4c+3) for the backward. */
int kgc_tail_apply(const float* pre, const float* stats, const float* gamma, const float* beta,
                   int64_t n_rows, int32_t Dout, float* all_ent, const int64_t* out_seed, float out_drop_p,
                   uint8_t* out_keep, void* stream);
/* Backward of the tail.  all_ent = tanh(BatchNorm(pre)) is recomputed from pre (one plane less to read).
 * kgc_tail_bwd_reduce: partial column sums of dz = g_ent*(1-all_ent^2) and dz*xhat; kgc_colsum_finalize -> sums[0] =
 * sum dz (= d beta), sums[1] = sum dz*xhat (= d gamma), all-reduced by a partitioned caller; kgc_tail_bwd_apply:
 * d_out[n_rows,Dout] = d_pre / 3 (BatchNorm backward over n_rows_global rows when training) - ONE plane: the self-loop
 * transform's upstream gradient as it is, the in / out halves' after the keep flags x 1/(1-p): applied by the GEMMs
 * (d_res_in = d_res_out = NULL), or written here as two more planes d_res_in / d_res_out [n_rows,Dout] from
 * kgc_tail_fwd's keep flags (keep NULL: no dropout, both planes = d_out; both planes or neither).  slot_h != NULL: plane h
 * is compacted (see kgc_tail_fwd) and receives only the rows that have edges, at their compact row. */
/* out_keep != NULL: the forward dropped its output (kgc_tail_apply): g_ent is taken x keep flag x out_scale = 1/(1-p). */
int kgc_tail_bwd_reduce(const float* g_ent, const float* pre, const float* stats, const float* gamma, const float* beta,
                        int64_t n_rows, int32_t Dout, double* partials, const uint8_t* out_keep, float out_scale,
                        void* stream);
int kgc_tail_bwd_apply(const float* g_ent, const float* pre, const float* stats, const float* gamma, const float* beta,
                       const double* sums, int32_t training, int64_t n_rows, int64_t n_rows_global, int32_t Dout,
                       float* d_out, const uint8_t* keep, float keep_scale, float* d_res_in, const int32_t* slot_in,
                       float* d_res_out, const int32_t* slot_out, const uint8_t* out_keep, float out_scale,
                       void* stream);

/* ---- K0: parameter-side work of one layer step, batched --------------------------------------------------
 * kgc_conv_prep (forward): relp = cat(rels, loop_rel) (model.py:86); all_rel = relp @ w_rel (model.py:107, all
 * n_rels + 1 rows - the caller drops the last); and the hi / lo TF32 packs kgc_gemm_nt_batch needs for the three
 * transforms of the step and of its backward: packed_fwd = 3 x pack(W_h as [K = D, N = Dout]), packed_bwd =
 * 4 x pack(W_h^T as [K = Dout, N = D]), h = in, out, loop, rel, each kgc_gemm_packed_b_bytes long, the self-loop weight
 * pre-scaled by loop_rel . loop_edge (model.py:92-94 folded: (x . lr . le) @ W = x @ diag(lr . le) W).
 * kgc_conv_param_grads (backward): from m_loop = x^T @ d_res_loop and the type-sorted edge reduction d_relp:
 *   d_w_loop = diag(lr . le) m_loop;  d_v = rowsum(m_loop . w_loop);  d_loop_edge = d_v . lr;
 *   d_relp' = d_relp + [g_rel; 0] @ w_rel^T;  d_rels = d_relp'[:-1];  d_loop_rel = d_v . le + d_relp'[-1];
 *   d_w_rel = relp^T @ [g_rel; 0]   (g_rel may be NULL: no gradient reached all_rel).
 * rel_add (optional, [n_rels, D]): the caller already holds g_rel @ w_rel^T (kgc_gemm_nt_batch with packed_bwd[3]) and has
 * written d_w_rel itself (kgc_gemm_tn_tc_batch) - the two products over the relation rows then run on the tensor cores instead of
 * this kernel's per-thread loops (0.29 ms at 1,644 relation rows).
 * Weights are contiguous [D, Dout]; D, Dout <= 256. */
int kgc_conv_prep(const float* rels, int32_t n_rels, const float* loop_rel, const float* loop_edge, const float* w_in,
                  const float* w_out, const float* w_loop, const float* w_rel, int32_t D, int32_t Dout, float* relp,
                  float* all_rel, float* packed_fwd, float* packed_bwd, void* stream);
int kgc_conv_param_grads(const float* m_loop, const float* w_loop, const float* loop_rel, const float* loop_edge,
                         const float* relp, const float* w_rel, const float* g_rel, const float* d_relp,
                         int32_t n_rels, int32_t D, int32_t Dout, float* d_w_loop, float* d_loop_rel,
                         float* d_loop_edge, float* d_rels, float* d_w_rel, const float* rel_add, void* stream);

/* ---- K4b: dense transforms on the tensor cores with fp32-grade accuracy (3xTF32) --------------------------
 * Replaces the fp32 matmuls of model.py:116 (x_j_rel @ W, after the aggregate-then-transform reordering
 * agg_h @ W_h) and of its autograd (d_res_h @ W_h^T):   C[M,N] = A[M,K] @ Bt[N,K]^T
 * A: fp32 row-major, leading dimension lda (a multiple of 4), streamed through TMA; C: fp32 row-major, 16-byte
 * aligned, leading dimension ldc (a multiple of 4), written by TMA stores; Bt: the small operand,
 * packed once per call by kgc_gemm_pack_b from B viewed as element (k, n) = B[k*stride_k + n*stride_n]
 * (hi / lo TF32 split, zero padded; size kgc_gemm_packed_b_bytes).  K <= 256, N <= 1024.
 * Every fp32 value v is split v = hi + lo (hi = top 19 bits); C = A_hi Bt_hi + A_lo Bt_hi + A_hi Bt_lo is
 * accumulated in fp32 by tcgen05.mma kind::tf32 - error ~2^-22 relative per product, i.e. fp32-level. */
size_t kgc_gemm_packed_b_bytes(int32_t N, int32_t K);
int kgc_gemm_pack_b(const float* B, int64_t stride_k, int64_t stride_n, int32_t N, int32_t K, float* packed,
                    void* stream);
/* n_prob (1..3) products of IDENTICAL shape in one launch (one product: n_prob = 1; the in / out / self-loop transforms
 * of a layer step: 3): A[i], packed_b[i], C[i] are HOST arrays of device pointers.  The CTAs are dealt to (problem, column
 * tile) groups.
 * keep (NULL: none) applies dropout to the streamed operand while it is split (backward of the layer tail, model.py:103):
 * kgc_tail_fwd's packed keep flags (byte c of row m = columns 4c..4c+3, rows keep_pitch bytes apart; problem 0 reads the
 * low nibble, problem 1 the high nibble, problem 2 takes the operand as it is); a kept element is multiplied by
 * keep_scale, a dropped one is 0.  The three problems may (and in the layer do) stream the SAME plane A[0] = A[1] = A[2]. */
int kgc_gemm_nt_batch(int32_t n_prob, const float* const* A, int64_t M, int32_t K, int64_t lda,
                      const float* const* packed_b, int32_t N, float* const* C, int64_t ldc, const uint8_t* keep,
                      int32_t keep_pitch, float keep_scale, void* stream);
/* Same kernel with the streamed operand AND the result transposed in memory (the long dimension M contiguous):
 *   Ct[n, m] = sum_k At[k, m] * Bt[n, k],  At: [K, M] row-major, pitch ldat;  Ct: [N, M] row-major, pitch ldct.
 * M % 32 == 0.  Used for the autograd of ConvE's fc layer (model.py:173): d_W[out, flat] = d_y^T @ x_flat and
 * d_x_flat[B, flat] = d_y @ W, where flat = 39,200 is the long dimension. */
int kgc_gemm_nt_trans(const float* At, int64_t M, int32_t K, int64_t ldat, const float* packed_b, int32_t N,
                      float* Ct, int64_t ldct, void* stream);

/* ---- K4c: weight-gradient reductions  C[Ka,Nb] = A[M,Ka]^T @ B[M,Nb]  (autograd of model.py:116 w.r.t. W) ----
 * Plain fp32 FMAs; every CTA reduces a slab of rows into a register-resident Ka x Nb partial, partials are added
 * in CTA order (deterministic).  Ka <= 128, Nb <= 256, all dimensions / leading dimensions multiples of 4. */
size_t kgc_gemm_tn_workspace_bytes(int64_t M, int32_t Ka, int32_t Nb);
int kgc_gemm_tn(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int32_t Ka, int32_t Nb,
                float* C, void* workspace, size_t workspace_bytes, void* stream);

/* Same product on the tensor cores (3xTF32, fp32-grade), see kgc_gemm_tn_tc_batch below. */
size_t kgc_gemm_tn_tc_workspace_bytes(int64_t M, int32_t Ka, int32_t Nb);

/* Split-K product of K-major operands with a LONG contraction (ConvE's fc forward, model.py:173: y[B, out] =
 * x_flat[B, flat] @ W[out, flat]^T, flat = 39,200):  C[Ma, Nb] = A[Ma, K] @ Bt[Nb, K]^T.  The K range is cut into
 * per-CTA slabs, both operands are streamed and split (3xTF32), partial products stay in TMEM and are added in CTA
 * order.  Ma <= 128, Nb <= 224, Nb / lda / ldb multiples of 4; workspace = kgc_gemm_tn_tc_workspace_bytes(K, Ma, Nb). */
int kgc_gemm_nt_splitk(const float* A, int64_t lda, const float* Bt, int64_t ldb, int64_t K, int32_t Ma, int32_t Nb,
                       float* C, void* workspace, size_t workspace_bytes, void* stream);

/* n_prob (1..3) weight-gradient reductions C[i] = A[i]^T @ B[i] of identical shape in one launch on the tensor cores
 * (3xTF32, fp32-grade; one reduction: n_prob = 1; d_W of the in / out / self-loop transforms: 3).  Both operands are
 * MN-major for the MMA (TMA boxes of 32 columns x 32 rows, 128-byte swizzle), both are split hi / lo in shared memory,
 * D[128 x Nb] stays in TMEM for the CTA's row slab; per-CTA partials are added in CTA order.  Ka <= 128, Nb <= 224,
 * multiples of 4.  A, B, C are HOST arrays of device pointers; the CTAs are dealt to (problem, row slab) pairs, so every
 * CTA sweeps a 3x longer slab than in three separate launches and three times fewer partials are added.  Workspace:
 * kgc_gemm_tn_tc_workspace_bytes(M, Ka, Nb) for any n_prob.
 * rows (NULL: M for every problem) = HOST array of rows[i] <= M rows in problem i (a compacted plane of the layer).  The
 * row slabs are those of M rows: a problem of M rows gets the bits it gets with rows = NULL; the others sum the slabs
 * their rows fill.
 * keep (NULL: none): the keep flags applied to the B operand (the upstream plane) while it is split, as in
 * kgc_gemm_nt_batch. */
int kgc_gemm_tn_tc_batch(int32_t n_prob, const float* const* A, int64_t lda, const float* const* B, int64_t ldb,
                         const int64_t* rows, int64_t M, int32_t Ka, int32_t Nb, float* const* C, void* workspace,
                         size_t workspace_bytes, const uint8_t* keep, int32_t keep_pitch, float keep_scale, void* stream);

/* ---- K5: label / batch builder ---------------------------------------------------------------------
 * Replaces KBDataset.get_label + label smoothing + collate (data_loader.py:25-51): for the batch's
 * query ids qid[B] (int64) and the query->objects CSR (ptr int64 [Q+1], idx int32 [nnz]):
 *   label[b, :] = add;  label[b, idx[k]] = pos   with the host passing pos = (1-ls)*1 + 1/N and
 *   add = 1/N when smoothing (data_loader.py:41-43), else pos = 1, add = 0.
 * triple_out[b,:] = triples[qid[b],:] (int64 [Q,3]). */
int kgc_label_build(const int64_t* qid, int64_t B, const int64_t* triples, const int64_t* ptr,
                    const int32_t* idx, int64_t n_entity, float pos, float add,
                    int64_t* triple_out, float* label, void* stream);

/* Extension with NO reference counterpart (the reference trains 1-N and ships no sampler,
 * SURVEY.md fact 2; "parity unpinned"): k negatives per query as a pure function of the caller's
 * uint32 draws.  neg[b,j] = first of draws[b,j,0..tries) mapped to [0,N) by (u * N) >> 32 that is
 * not a positive of query qid[b]; -1 if every try collides. */
int kgc_neg_sample(const int64_t* qid, int64_t B, const int64_t* ptr, const int32_t* idx, int64_t n_entity,
                   const uint32_t* draws, int32_t k, int32_t tries, int32_t* neg, void* stream);

/* Positive sampler, the companion of kgc_neg_sample (extension): out[b, j] = idx[ptr[q] + ((draws[b, j] * len_q) >> 32)]
 * with q = qid[b] and len_q = ptr[q + 1] - ptr[q] - sampling with replacement from the query's object list; -1 for a
 * query without objects.  A pure function of the caller's uint32 draws [B, p]; out int32 [B, p]. */
int kgc_pos_sample(const int64_t* qid, int64_t B, const int64_t* ptr, const int32_t* idx, const uint32_t* draws,
                   int32_t p, int32_t* out, void* stream);

/* Edge sampler, likewise an extension without a reference counterpart (the reference always convolves over the full
 * edge list built at data_loader.py:132-157).  m triples drawn with replacement, t_j = (draws[j] * n_triples) >> 32; the
 * sampled sub-graph keeps the reference's layout: columns 0..m-1 = in-half edges t_j, m..2m-1 = their reverses
 * t_j + n_triples.  src / dst / type = the rows of edge_index and edge_attr[0] (int64 [2 n_triples]); outputs int64 [2m];
 * eids = the chosen columns (the rows of edge_embeddings the sub-graph uses). */
int kgc_edge_sample(const int64_t* src, const int64_t* dst, const int64_t* type, int64_t n_triples, const uint32_t* draws,
                    int64_t m, int64_t* sub_src, int64_t* sub_dst, int64_t* sub_type, int64_t* eids, void* stream);

/* ---- K7: ConvE feature-map normalisation: BatchNorm2d (+ ReLU) + feature dropout (SURVEY "next" row N2) --------
 * Replaces model.py:168-170 (x = bn1(x); x = relu(x); x = feature_drop(x)) on the [B, C, H, W] convolution output
 * (HW = H * W, a multiple of 4; contiguous) and its autograd; with relu = 0 and drop_p = 0 also bn0 (model.py:165),
 * the ONE-channel BatchNorm2d over the [B, 1, 2 k_w, k_h] input image, which cuDNN gives to a single CTA.
 * Forward: training != 0 -> batch statistics (fp64 accumulation, fixed-order reduction) + the running-statistics
 * update of nn.BatchNorm2d (momentum, unbiased variance; running_* may be NULL); else the running statistics.
 * stats[2][C] = {mean, rstd} is written for the backward.  Dropout (training only, drop_p in [0, 1)): keep mask from a
 * Philox4x32-10 stream keyed by *seed (device int64), regenerated by the backward - no mask tensor.
 * Backward: dx; sums[2][C] = {d_beta, d_gamma}.  partials: kgc_bn2d_partials_bytes(C) of scratch. */
size_t kgc_bn2d_partials_bytes(int32_t C);
int kgc_bn2d_relu_drop_fwd(const float* x, int64_t B, int32_t C, int32_t HW, const float* gamma, const float* beta,
                           float* running_mean, float* running_var, float eps, float momentum, int32_t training,
                           int32_t relu, const int64_t* seed, float drop_p, double* partials, float* stats, float* y,
                           void* stream);
int kgc_bn2d_relu_drop_bwd(const float* dy, const float* x, int64_t B, int32_t C, int32_t HW, const float* gamma,
                           const float* beta, const float* stats, int32_t training, int32_t relu, const int64_t* seed,
                           float drop_p, double* partials, float* sums, float* dx, void* stream);

/* ---- K8: ConvE's one-input-channel convolution (SURVEY "next" row N2) ------------------------------------------
 * Replaces model.py:166 (x = self.conv_e(x): nn.Conv2d(1, F, (K, K), stride 1, padding 0)) and its autograd.
 * torch layouts, contiguous fp32: x [B, 1, H, W], w [F, 1, K, K], bias [F] or NULL, y / dy [B, F, H-K+1, W-K+1].
 * Direct fp32 FMA kernels, fixed summation order (deterministic).  kgc_conv1ch_supported: W = 20, K in {3, 5, 7},
 * K <= H <= 64 and the filters fit shared memory; callers use the library convolution otherwise.
 * Backward: dx [B, 1, H, W] and/or dw [F, 1, K, K] (either may be NULL); workspace: kgc_conv1ch_bwd_workspace_bytes. */
int kgc_conv1ch_supported(int32_t F, int32_t K, int32_t H, int32_t W);
size_t kgc_conv1ch_bwd_workspace_bytes(int64_t B, int32_t F, int32_t K);
int kgc_conv1ch_fwd(const float* x, const float* w, const float* bias, int64_t B, int32_t F, int32_t K, int32_t H,
                    int32_t W, float* y, void* stream);
int kgc_conv1ch_bwd(const float* dy, const float* x, const float* w, int64_t B, int32_t F, int32_t K, int32_t H,
                    int32_t W, float* dx, float* dw, void* workspace, void* stream);

/* ---- K9: gradient-norm clipping + Adam (the optimiser half of the training step, main.py:68-71, 217) --------------
 * One call = nn.utils.clip_grad_norm_(params, max_norm) followed by torch.optim.Adam.step() (amsgrad off, L2 weight
 * decay) over fp32 tensors: squared-norm partials (fp64, fixed order), coefficient + step counter + bias corrections on the
 * device, then the update with coef * g applied in flight (gradients are not modified).
 * tensors[n]: device table; items[n_items][4] int32 = {tensor, chunk, elements in chunk (<= kgc_opt_chunk_elems()), 0};
 * hyper[6] (device fp32) = lr, beta1, beta2, eps, weight_decay, max_norm (<= 0: no clipping); state[5] (device fp64) =
 * step count (in/out), clip coefficient, lr / (1 - b1^t), 1 / sqrt(1 - b2^t), gradient norm (out); partials[n_items]. */
typedef struct { float* param; const float* grad; float* exp_avg; float* exp_avg_sq; } kgc_opt_tensor_t;
int32_t kgc_opt_chunk_elems(void);
int kgc_clip_adam_step(const kgc_opt_tensor_t* tensors, const int32_t* items, int64_t n_items, const float* hyper,
                       double* state, double* partials, void* stream);
/* The same step split in two for a model sharded over several GPUs (each rank holds some tensors, or some rows of them):
 * kgc_clip_adam_sqnorm writes sqnorm[0] (device fp64) = the squared norm of this rank's items, where an item whose 4th
 * field is non-zero adds 0 (a replicated tensor that another rank counts); the caller sums sqnorm over the ranks and
 * kgc_clip_adam_apply runs the step's coefficient and update kernels with the norm sqrt(sqnorm[0]).  On one rank without
 * flags the two calls equal kgc_clip_adam_step bit for bit.  partials[n_items] as above; the step ignores the 4th field. */
int kgc_clip_adam_sqnorm(const kgc_opt_tensor_t* tensors, const int32_t* items, int64_t n_items, double* partials,
                         double* sqnorm, void* stream);
int kgc_clip_adam_apply(const kgc_opt_tensor_t* tensors, const int32_t* items, int64_t n_items, const float* hyper,
                        double* state, const double* sqnorm, void* stream);

/* ---- K10: halo exchange of the dst-partitioned layer over NVLink peer memory (SURVEY.md 8(e)) -----------------
 * Replaces the library all-gather of x / reduce-scatter of d_x of the partitioned layer: every rank keeps the gathered
 * node table and its partial d_x in SYMMETRIC buffers (same size on every rank, peer-mapped); *_ptrs_dev = device array
 * of `world` pointers to the ranks' buffers.
 *   kgc_p2p_barrier      flag barrier: flag_ptrs_dev[r] = rank r's uint32[world] flag array (zero-initialised);
 *                        *epoch (local, zero-initialised) counts barriers; no data-path time-out: a ~2 minute watchdog sets
 *                        *error = 1 and traps.  Barriers issued on different streams need their own flag array + epoch.
 *   kgc_p2p_halo_gather  every rank's node table = its own block_rows rows, then its halo.  Pulls the remote rows
 *                        rows[n_rows] (renumbered ids: owner g / block_rows, local row g % block_rows) from the head of
 *                        their owners' tables into rows block_rows + i of this rank's table.  order (optional): a permutation of
 *                        the list positions = the sequence in which they are pulled (spreads every reader over all owners).
 *   kgc_p2p_halo_reduce  out[v] = addend[v] + sum over the ranks r with idx[r * n_rows + j] >= 0, in ascending r, of
 *                        row idx[r * n_rows + j] of part_r   (deterministic); v = j for all j < n_rows (row_ids NULL: every
 *                        row of this rank) or v = row_ids[j] (only the rows other ranks contributed to); addend == out
 *                        is allowed (in-place add of the remote partials).
 *   kgc_p2p_allreduce    one-shot sum of a small vector (n_bytes, a multiple of 16; fp32 or fp64) over the ranks: copy
 *                        into this rank's staging slot (stage_ptrs_dev[r] + offset_bytes), flag barrier, every rank adds
 *                        all slots in rank order (identical bits everywhere).  in == out is allowed.  One CTA up to 64 KB
 *                        (BatchNorm sums, split hub rows); wider payloads (the replicated-parameter gradients, ~1 MB)
 *                        stage / meet / add in three launches with many CTAs. */
int kgc_p2p_allreduce(void* const* stage_ptrs_dev, int64_t offset_bytes, void* const* flag_ptrs_dev, int32_t rank,
                      int32_t world, uint32_t* epoch, int32_t* error, const void* in, void* out, int64_t n_bytes,
                      int32_t is_double, void* stream);
int kgc_p2p_barrier(void* const* flag_ptrs_dev, int32_t rank, int32_t world, uint32_t* epoch, int32_t* error, void* stream);
int kgc_p2p_halo_gather(void* const* table_ptrs_dev, int32_t rank, const int32_t* rows, const int32_t* order, int64_t n_rows,
                        int64_t block_rows, int32_t D, void* stream);
int kgc_p2p_halo_reduce(void* const* part_ptrs_dev, int32_t world, const int32_t* idx, const int32_t* row_ids, int64_t n_rows,
                        const float* addend, float* out, int32_t D, void* stream);

/* ---- N4: native text -> id ingest (host C++, no device code; SURVEY "next" row N4) ---------------------------------
 * Replaces the two per-line passes of DataLoader._load_data (data_loader.py:64-111) over <data_dir>/{train,valid,test}.txt:
 * ids in first-appearance order (tokens lower-cased for the vocabulary, looked up as written - the reference's quirk),
 * triple arrays, and the (s, r) -> objects / (o, r + R) -> subjects groups as CSR query sets in the reference's order
 * (train: one query per group created during the train split, in creation order, train-only objects; valid / test:
 * one tail and one head query per triple with the objects of ALL splits; objects sorted and unique).
 * kgc_ingest_open: 0 OK; 1 malformed line (not three tokens); 2 unsupported text (non-ASCII token, relation ending in
 * "_reverse": the caller runs the reference's Python passes); 3 I/O; 4 unknown token at look-up (kgc_last_error() is the
 * token: the reference raises KeyError).
 * Query set q: 0 train, 1 valid_tail, 2 valid_head, 3 test_tail, 4 test_head.  Train: ptr / idx are per query.  Valid / test:
 * the object lists are stored ONCE per (s, r) group the set references (ptr / idx over groups) plus query -> group, because
 * a hub group is the filter of thousands of queries.
 * kgc_ingest_count what: 0 entities, 1 relations R, 2/3/4 triples of train / valid / test, 5/6 bytes of the entity /
 * relation token blobs, 10 + 2q queries and 11 + 2q stored label entries of set q, 20 + q rows of its ptr array.
 * kgc_ingest_copy array: 5/6 all entity / relation tokens in id order, each followed by '\n'; 2/3/4 split triples int64 [n,3];
 * 10 + 3q query triples int64 [Q,3] (train: o = -1), 11 + 3q ptr int64 [rows+1], 12 + 3q idx int32, 30 + q query -> group
 * int32 [Q] (valid / test).  kgc_ingest_name kind: 0 entity, 1 relation token (lower-cased) of an id. */
typedef struct kgc_ingest kgc_ingest_t;
int kgc_ingest_open(const char* data_dir, kgc_ingest_t** out);
void kgc_ingest_close(kgc_ingest_t* h);
int64_t kgc_ingest_count(const kgc_ingest_t* h, int32_t what);
int kgc_ingest_copy(const kgc_ingest_t* h, int32_t array, void* dst, int64_t capacity_bytes);
const char* kgc_ingest_name(const kgc_ingest_t* h, int32_t kind, int64_t id);

/* ---- K6t: 1-N scoring in TRAINING (dense [B,N] sigmoid scores and their autograd) -------------------------
 * Replaces model.py:177-179 (x = mm(x, all_ent^T); x += bias; sigmoid) where the caller needs the dense matrix
 * (BCE against the multi-hot label, main.py:63-66).  Forward: the K4b tensor-core kernel (3xTF32, fp32-grade) with
 * the entity table E[n_ent, D] as the streamed operand and the queries X[B, D] as the packed small one
 * (kgc_gemm_pack_b with stride_k = 1, stride_n = ld_x); the epilogue adds bias[n], applies the logistic sigmoid and
 * TMA-stores the block transposed:  pred[b, n] = sigmoid(X[b,:] . E[n,:] + bias[n]),  pred row pitch ld_pred
 * (a multiple of 4, >= n_ent; 16-byte aligned).  D <= 256, D % 4 == 0, B <= 1024.
 * Backward through the sigmoid: d_logitT[n, b] = d_pred[b, n] * pred[b, n] * (1 - pred[b, n]) written TRANSPOSED
 * ([n_ent, ldt], ldt >= B, columns [B, ldt) zeroed) so that d_X = kgc_gemm_tn_tc_batch(d_logitT, E) and
 * d_E = kgc_gemm_nt_batch(d_logitT, X) stream it row-major; d_bias[n] = sum_b d_logitT[n, b] in a fixed order. */
int kgc_score_1n_fwd(const float* ent, int64_t n_ent, int32_t D, int64_t ld_ent, const float* packed_x, int32_t B,
                     const float* bias, float* pred, int64_t ld_pred, void* stream);
/* The same product without the sigmoid: logits[b, n] = X[b,:] . E[n,:] + bias[n] (fp32-grade).  Exact-mode evaluation
 * (main.py:121-126 ranks fp32 scores; the fused bf16 scorer K6 can move a rank between two entities whose logits lie
 * within 2^-7 relative of each other): rank on these with kgc_rank_count_dense + kgc_rank_finalize. */
int kgc_score_1n_logits(const float* ent, int64_t n_ent, int32_t D, int64_t ld_ent, const float* packed_x, int32_t B,
                        const float* bias, float* logits, int64_t ld_logits, void* stream);
int kgc_score_1n_bwd_logit(const float* d_pred, int64_t ld_dp, const float* pred, int64_t ld_p, int64_t n_ent,
                           int32_t B, int32_t ldt, float* d_logitT, float* d_bias, void* stream);

/* ---- N1: training loss against SPARSE positives (SURVEY.md 8(f) row N1) ------------------------------------------
 * Replaces the dense label build (data_loader.py:34-43), its host-to-device copy (main.py:60), BCELoss (model.py:42-44,
 * main.py:62) and the loss's backward down to the logit gradient, for the batch's query ids and the query->objects CSR
 * that kgc_label_build takes.  kgc_score_1n_fwd_t stores predT[n, b] = sigmoid(logit) (rows of ldt >= B floats,
 * ldt % 4 == 0) - the scorer's natural orientation; kgc_label_mask_t_build keeps the positives as bits per ENTITY
 * (mask_t [n_entity, ceil(B / 32)] uint32, zeroed by the call): bit (b & 31) of word (b >> 5) of row j is set for every
 * positive j of query qid[b].  kgc_bce_1n_bwd_logit_t, with y[b, n] = pos where the bit is set, add elsewhere, and
 * p = predT[n, b], makes one row-wise pass that OVERWRITES pred_t with the transposed logit gradient:
 *   loss[0]        = mean_{b,n} ((y - 1) * max(log1p(-p), -100) - y * max(log(p), -100))       (torch BCELoss, mean)
 *   predT[n, b]   <- (p - y) / max((1 - p) p, 1e-12) / (B N) * p * (1 - p)   (columns [B, ldt) zeroed)
 *   d_bias[n]      = sum_b predT[n, b]
 * i.e. the gradient of the loss for a unit upstream gradient, in the layout kgc_score_1n_bwd_logit produces.
 * loss_partial: kgc_bce_1n_t_blocks(n_ent) doubles of workspace; sums are formed in a fixed order (deterministic).
 * Entity-major because [B, N] row pitches of 4 N bytes made batch-major kernels move their 2.35 GB in 128-byte pieces,
 * one per DRAM page (3.4 ms each at N = 4.6 M). */
int kgc_score_1n_fwd_t(const float* ent, int64_t n_ent, int32_t D, int64_t ld_ent, const float* packed_x, int32_t B,
                       const float* bias, float* pred_t, int64_t ld_t, void* stream);
int64_t kgc_bce_1n_t_blocks(int64_t n_ent);
int kgc_label_mask_t_build(const int64_t* qid, int64_t B, const int64_t* ptr, const int32_t* idx, int64_t n_entity,
                           uint32_t* mask_t, void* stream);
int kgc_bce_1n_bwd_logit_t(float* pred_t, const uint32_t* mask_t, int64_t n_ent, int32_t B, int32_t ldt, float pos, float add,
                           float* d_bias, double* loss_partial, float* loss, void* stream);
/* The same loss on an entity-sharded table (MGCN.shard: each GPU holds the rows of the entities it owns, in its own order).
 * kgc_label_mask_t_build_rows: kgc_label_mask_t_build with positive j's bit set in row row_of[j] of mask_t [n_rows,
 * ceil(B / 32)] (zeroed by the call); row_of [n_entity] int32 maps a global id to its local row, -1 when another rank owns
 * it (every id in idx must index row_of).  kgc_bce_1n_bwd_logit_t_shard: kgc_bce_1n_bwd_logit_t's pass over the n_rows
 * local rows with the divisor of the whole table, B * n_total (formed as the unsharded call forms B * n_ent), so every
 * gradient row and d_bias entry is bit-identical to that entity's row of the unsharded call; instead of the mean it writes
 * the shard's fp64 sum of the loss terms, in a fixed order, to loss_sum[0] (device).  loss_partial:
 * kgc_bce_1n_t_blocks(n_rows) doubles. */
int kgc_label_mask_t_build_rows(const int64_t* qid, int64_t B, const int64_t* ptr, const int32_t* idx, const int32_t* row_of,
                                int64_t n_rows, uint32_t* mask_t, void* stream);
int kgc_bce_1n_bwd_logit_t_shard(float* pred_t, const uint32_t* mask_t, int64_t n_rows, int32_t B, int32_t ldt, float pos,
                                 float add, int64_t n_total, float* d_bias, double* loss_partial, double* loss_sum,
                                 void* stream);

/* ---- K6: fused 1-N scoring + filter + rank (tcgen05 / TMA) --------------------------------------------
 * Replaces model.py:177-178 (X @ all_ent^T + bias) and main.py:122-126 (filter, rank) without
 * materialising the [B,N] score matrix.  Ranking is on the logit (sigmoid is monotone and saturates,
 * SURVEY.md section 7 "Tie semantics").
 *   kpad = kgc_score_kpad(d): padded K (multiple of 16, >= d + 3, <= 256; 208 for d = 200), -1 if d is too large.
 *   kgc_score_pack_*: fp32 rows -> bf16 rows of pitch kpad with the bias folded into three extra K columns
 *     (entity side: bf16 hi/mid/lo split of bias[j]; query side: 1, 1, 1), zero padded.
 *   kgc_score_rank: for every query q, ADD to count_gt[q] the number of entities j in [0, n) with
 *     s[q,j] > thr[q] (and to count_eq[q], when not NULL, those with s == thr), s being the
 *     bf16 x bf16 -> fp32 tensor-core product.  The caller zeroes the counters; entity-sharded callers
 *     call it once per shard and all-reduce the integers.
 *   kgc_score_pairs: s for explicit (query row, entity row) pairs through the SAME MMA path (the target
 *     score thr[q] and the scores of the filtered positives), so the correction below is bit-consistent.
 *   kgc_rank_finalize (main.py:122-133): ranks[q] = 1 + count_gt[q] - #{k in filter(q), idx[k] != obj[q],
 *     s_filt[k] > thr[q]}; eq_out likewise (minus the target itself); sums13 = {count, sum rank,
 *     sum 1/rank (fp32 division as main.py:131), hits@1..10} reduced in a fixed order. */
int32_t kgc_score_kpad(int32_t d);
int kgc_score_pack_entities(const float* all_ent, const float* bias, int64_t n, int32_t d,
                            uint16_t* e_bf16, void* stream);
int kgc_score_pack_queries(const float* xq, int64_t b, int32_t d, uint16_t* q_bf16, void* stream);
size_t kgc_score_pairs_workspace_bytes(int64_t n_pairs, int32_t kpad);
int kgc_score_pairs(const uint16_t* q_bf16, const uint16_t* e_bf16, const int32_t* pair_q, const int32_t* pair_e,
                    int64_t n_pairs, int32_t kpad, float* s_out, void* workspace, size_t workspace_bytes,
                    void* stream);
int kgc_score_rank(const uint16_t* q_bf16, const uint16_t* e_bf16, int64_t b, int64_t n, int32_t kpad,
                   const float* thr, int32_t* count_gt, int32_t* count_eq, void* stream);
/* Exact-mode counts over DENSE fp32 logits [b, ld] (kgc_score_1n_logits): count_gt[q] += #{j < n_ent : logit[q,j] > thr[q]},
 * count_eq likewise (may be NULL); caller zeroes the counters; integer atomics only.  b <= 65,535 per call. */
int kgc_rank_count_dense(const float* logits, int64_t ld, int64_t n_ent, int64_t b, const float* thr,
                         int32_t* count_gt, int32_t* count_eq, void* stream);
int kgc_rank_finalize(const int32_t* count_gt, const int32_t* count_eq, const float* thr, const float* s_filt,
                      const int64_t* filt_ptr, const int32_t* filt_idx, const int64_t* obj, int64_t b,
                      int32_t* ranks, int32_t* eq_out, double* sums13, void* stream);

/* ---- K6k: filtered top-k entity prediction -------------------------------------------------------------
 * For every query q, the k best ELIGIBLE entities: j in [0, n) not in q's exclusion list, ordered by (logit descending,
 * entity id ascending), -0.0 equal to +0.0.  excl_ptr [b+1] int64 / excl_idx int32: the exclusion CSR, each row sorted
 * ascending (duplicates allowed, ids outside [0, n) ignored); both NULL: no filter.  1 <= k <= 32.
 * Output: top_s [b, k] logits, top_id [b, k], count [b] = number of real entries; rows with fewer than k eligible
 * entities are padded with (-inf, -1).  Deterministic (no float atomics): repeated calls are bit-identical.
 *   kgc_score_topk: the K6 sweep (same TMA / tcgen05 path and bf16 operands as kgc_score_rank and kgc_score_pairs, so
 *     top_s[q, i] equals kgc_score_pairs of (q, top_id[q, i]) bit for bit) with a register-resident top-k epilogue; each
 *     work item writes its partial list to the workspace, a merge kernel reduces them.  Items skip candidates below the
 *     K-th score another item of the same query already found (integer max), which does not change the result.
 *   kgc_topk_dense: the same selection over DENSE fp32 logits [b, ld] (kgc_score_1n_logits, exact mode); b <= 65,535.
 * workspace: at least the matching *_workspace_bytes (0 for arguments the call rejects), device memory, 16-byte aligned. */
size_t kgc_score_topk_workspace_bytes(int64_t b, int64_t n, int32_t kpad, int32_t k);
int kgc_score_topk(const uint16_t* q_bf16, const uint16_t* e_bf16, int64_t b, int64_t n, int32_t kpad,
                   const int64_t* excl_ptr, const int32_t* excl_idx, int32_t k, float* top_s, int32_t* top_id,
                   int32_t* count, void* workspace, size_t workspace_bytes, void* stream);
size_t kgc_topk_dense_workspace_bytes(int64_t b, int64_t n, int32_t k);
int kgc_topk_dense(const float* logits, int64_t ld, int64_t n, int64_t b, const int64_t* excl_ptr,
                   const int32_t* excl_idx, int32_t k, float* top_s, int32_t* top_id, int32_t* count,
                   void* workspace, size_t workspace_bytes, void* stream);
/* kgc_topk_merge: the k best entries of the union of n_lists finished results, e.g. one per entity shard.
 * part_s [n_lists, b, k] float / part_id [n_lists, b, k] int32: each [k] row sorted as kgc_score_topk returns it
 * (logit descending, id ascending), ids < 0 padding; ids must be disjoint across lists (shards own disjoint rows).
 * Output as above: top_s / top_id [b, k] ordered by (logit descending, id ascending), -0.0 equal to +0.0, padded with
 * (-inf, -1); count [b] real entries.  Keys are unique, so the result does not depend on the list order.
 * n_lists >= 1, 0 < b < 2^31, 1 <= k <= 32.  One kernel, no workspace; deterministic. */
int kgc_topk_merge(const float* part_s, const int32_t* part_id, int64_t n_lists, int64_t b, int32_t k,
                   float* top_s, int32_t* top_id, int32_t* count, void* stream);

/* K6s: sampled (1-vs-k) scoring fused with the BCE loss (extension: negative-sampled training).  Query b scores the C
 * candidates cand[b, 0..C) (int32 [B, C]): the first n_pos carry the label pos, the rest add; an id outside [0, n_ent) is
 * an empty slot (no loss, no gradient).  x [B, D] contiguous, ent [n_ent, D] with row pitch ld_ent, bias [n_ent];
 * D % 4 == 0, D <= 256; x, ent, d_x 16-byte aligned.
 * kgc_sampled_bce_fwd, in one pass: loss[0] = mean over the valid slots of ATen's BCE of p = sigmoid(<x[b], ent[c]> +
 * bias[c]) (0 when no slot is valid), count[0] = the number of valid slots, g [B, C] = the logit gradient for a unit
 * upstream gradient (0 on empty slots, kgc_bce_1n_bwd_logit_t's formulas, csrc/bce.cuh, with the valid-slot count as divisor) and
 * d_x [B, D] = sum_c g[b, c] * ent[cand[b, c]] in slot order.  loss_partial: kgc_sampled_bce_fwd_blocks(B) doubles.
 * kgc_sampled_bce_bwd_table: the dense table gradient for the upstream scalar *scale (device memory):
 * d_ent[n] = sum over the slots s with cand[s] = n of g[s] * (*scale * x[b(s)]), d_bias[n] = *scale * sum g[s], in slot
 * order; rows no slot names are zero (d_ent [n_ent, D] with row pitch ld_d).  The (entity, slot) pairs are
 * stable-sorted by entity, no float atomics.  workspace: kgc_sampled_bce_bwd_table_workspace_bytes(B * C, n_ent) bytes.
 * Both deterministic, no host synchronisation (graph-capturable). */
int64_t kgc_sampled_bce_fwd_blocks(int64_t B);
int kgc_sampled_bce_fwd(const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                        const float* bias, const int32_t* cand, int32_t C, int32_t n_pos, float pos, float add,
                        float* g, float* d_x, int32_t* count, double* loss_partial, float* loss, void* stream);
/* kgc_sampled_adv_fwd: the same pass with self-adversarial negative weights (Sun et al. 2019, RotatE) at temperature
 * alpha = `temperature` (finite, >= 0; 0 gives uniform weights).  With P_b / Q_b the valid positive / negative slots of
 * query b, z its logits, l ATen's BCE term and w[b, j] = softmax over j in Q_b of (alpha z[b, j]) (a constant, no
 * gradient through it):
 *   loss[0] = 1/2 (1/Q+) sum_{b: P_b non-empty} (1/|P_b|) sum_{P_b} l(z, pos) + 1/2 (1/Q-) sum_{b: Q_b non-empty} sum_{Q_b} w l(z, add)
 * (a half whose count is 0 adds 0).  counts[0] = Q+, counts[1] = Q- (the numbers of queries with a valid positive /
 * negative slot).  g [B, C] = the logit gradient for a unit upstream gradient: c * (p - y) / max((1 - p) p, 1e-12) *
 * p (1 - p) with c = 1 / (2 Q+ |P_b|) on a positive slot, w / (2 Q-) on a negative one, 0 on empty slots.  d_x [B, D] =
 * sum_c g[b, c] * ent[cand[b, c]] (up to rounding: the negative part is summed online and rescaled as the running max
 * of alpha z rises).  loss_partial: 2 * kgc_sampled_bce_fwd_blocks(B) doubles.  Every candidate row is read once.  The
 * table gradient is kgc_sampled_bce_bwd_table on this g.  Deterministic, no host synchronisation (graph-capturable). */
int kgc_sampled_adv_fwd(const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                        const float* bias, const int32_t* cand, int32_t C, int32_t n_pos, float pos, float add,
                        float temperature, float* g, float* d_x, int32_t* counts, double* loss_partial, float* loss,
                        void* stream);
/* kgc_sampled_ce_fwd: the same pass with the softmax cross-entropy of each positive against its query's negatives
 * (InfoNCE; LibKGE's `kl`, PyKEEN's CrossEntropyLoss) at label smoothing eps = `label_smoothing` (in [0, 1]; pos and add
 * do not enter).  With P_b / Q_b the valid positive / negative slots of query b, z its logits, K_b = 1 + |Q_b| and, for
 * each p in P_b, the classes {p} u Q_b (duplicates count as separate classes; the other positives are not in p's
 * denominator), LSE_p = log(exp(z_p) + sum_{Q_b} exp(z_q)):
 *   l_p = (1 - eps) (LSE_p - z_p) + eps (LSE_p - (z_p + sum_{Q_b} z_q) / K_b),  loss[0] = (1/P) sum_b sum_{P_b} l_p
 * with P = count[0] = the number of valid positive slots (loss 0 when P = 0): cross_entropy(label_smoothing=eps) of
 * the row [z_p, z_{Q_b}] with target 0, averaged over the valid positive slots.  g [B, C] = the logit gradient for a
 * unit upstream gradient: (softmax_p(p) - (1 - eps) - eps / K_b) / P on a positive slot, sum_{P_b} (softmax_p(q) -
 * eps / K_b) / P on a negative one (softmax_p(q) = exp(z_q) / (exp(z_p) + sum_{Q_b} exp(z_q))), 0 on empty slots; a
 * positive without a valid negative adds 0 loss and 0 gradient.  d_x [B, D] = sum_c g[b, c] * ent[cand[b, c]] (up to
 * rounding: the negative part is summed online against the running max of z).  The log-sum-exp is taken against that
 * max, so no logit overflows.  loss_partial: kgc_sampled_bce_fwd_blocks(B) doubles.  Every negative row is read once,
 * the positive rows twice.  The table gradient is kgc_sampled_bce_bwd_table on this g.  Deterministic, no host
 * synchronisation (graph-capturable). */
int kgc_sampled_ce_fwd(const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                       const float* bias, const int32_t* cand, int32_t C, int32_t n_pos, float label_smoothing,
                       float* g, float* d_x, int32_t* count, double* loss_partial, float* loss, void* stream);
size_t kgc_sampled_bce_bwd_table_workspace_bytes(int64_t n_slots, int64_t n_ent);
int kgc_sampled_bce_bwd_table(const float* x, int64_t B, int32_t D, const int32_t* cand, int32_t C, const float* g,
                              const float* scale, int64_t n_ent, float* d_ent, int64_t ld_d, float* d_bias,
                              void* workspace, size_t workspace_bytes, void* stream);

/* K6s, shared negatives: every query of the batch scores the same k negatives shared [k] (int32) besides its own n_pos
 * positives pos_cand [B, n_pos] (n_pos >= 1).  The loss is the per-query loss above (kgc_sampled_*_fwd) on the broadcast
 * candidate matrix cand[b] = [pos_cand[b] | shared, with every entry that is a known object of query qid[b] (the
 * query->objects CSR of kgc_label_mask_t_build) set to -1]: the same value, gradients, divisors and empty-slot rules.
 * Duplicates in shared are separate slots; a filtered entry is an empty slot of that query only; an id outside
 * [0, n_ent) is an empty slot of every query.
 *   kgc_score_1n_logits_t: logitT[n, b] = E[n,:] . X[b,:] + bias[n] (fp32-grade, 3xTF32), kgc_score_1n_fwd_t without
 *     the sigmoid; here on E = the gathered shared rows.
 *   kgc_shared_rows: rows [k, D] contiguous = ent[shared], row_bias [k] = bias[shared] (zeros for an invalid id).
 *   kgc_shared_mask_build: mask_t [k, ceil(B / 32)] uint32, bit (b & 31) of word (b >> 5) of row j set iff shared[j] is
 *     a known object of query qid[b] (zeroed by the call); sorted_ids / sorted_slots [k]: the (id, slot) pairs
 *     stable-sorted by id (an invalid id sorts as n_ent), which kgc_shared_bwd_table takes.  CUB radix sort and a binary
 *     search per known object, integer operations only.  workspace: kgc_shared_mask_workspace_bytes(k, n_ent).
 *   kgc_shared_{bce,adv,ce}_loss: over logit_t [k, ldt] (ldt >= B; the shared logits of query b in column b), the mask
 *     and the positives: loss[0]; the logit gradient for a unit upstream gradient OVER logit_t (0 on filtered and empty
 *     slots and in columns [B, ldt) of the CTAs' 32-query groups); g_pos [B, n_pos], the positive slots' gradient;
 *     d_x [B, D] = sum_c g_pos[b, c] ent[pos_cand[b, c]] in slot order (the negatives' part is the caller's product of
 *     the gradient tile with the shared rows); d_bias_s [k] = sum_b of the gradient tile's row j, the CTAs' partials
 *     added in a fixed order.  The adversarial weights and the cross-entropy's log-sum-exp are per query over its k
 *     shared slots against their max.  workspace: kgc_shared_loss_workspace_bytes(B, k).
 *   kgc_shared_bwd_table: d_ent[n] += *scale * sum over the slots j with shared[j] = n of d_rows[j] (rows of pitch
 *     ld_rows), d_bias[n] += *scale * sum d_row_bias[j], added in slot order through the sorted pairs (no float atomics);
 *     the positives' part and the zero fill come first from kgc_sampled_bce_bwd_table on (pos_cand, g_pos).
 * All deterministic, no host synchronisation (graph-capturable). */
int kgc_score_1n_logits_t(const float* ent, int64_t n_ent, int32_t D, int64_t ld_ent, const float* packed_x, int32_t B,
                          const float* bias, float* logit_t, int64_t ld_t, void* stream);
int kgc_shared_rows(const float* ent, int64_t n_ent, int32_t D, int64_t ld_ent, const float* bias, const int32_t* shared,
                    int32_t k, float* rows, float* row_bias, void* stream);
size_t kgc_shared_mask_workspace_bytes(int32_t k, int64_t n_ent);
int kgc_shared_mask_build(const int32_t* shared, int32_t k, const int64_t* qid, int64_t B, const int64_t* ptr,
                          const int32_t* idx, int64_t n_ent, uint32_t* mask_t, int32_t* sorted_ids, int32_t* sorted_slots,
                          void* workspace, size_t workspace_bytes, void* stream);
int64_t kgc_shared_loss_blocks(int64_t B);
size_t kgc_shared_loss_workspace_bytes(int64_t B, int32_t k);
int kgc_shared_bce_loss(float* logit_t, int64_t ldt, const uint32_t* mask_t, const int32_t* shared, int32_t k,
                        const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                        const float* bias, const int32_t* pos_cand, int32_t n_pos, float pos, float add, float* g_pos,
                        float* d_x, float* d_bias_s, float* loss, void* workspace, size_t workspace_bytes, void* stream);
int kgc_shared_adv_loss(float* logit_t, int64_t ldt, const uint32_t* mask_t, const int32_t* shared, int32_t k,
                        const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                        const float* bias, const int32_t* pos_cand, int32_t n_pos, float pos, float add, float temperature,
                        float* g_pos, float* d_x, float* d_bias_s, float* loss, void* workspace, size_t workspace_bytes,
                        void* stream);
int kgc_shared_ce_loss(float* logit_t, int64_t ldt, const uint32_t* mask_t, const int32_t* shared, int32_t k,
                       const float* x, int64_t B, int32_t D, const float* ent, int64_t n_ent, int64_t ld_ent,
                       const float* bias, const int32_t* pos_cand, int32_t n_pos, float label_smoothing, float* g_pos,
                       float* d_x, float* d_bias_s, float* loss, void* workspace, size_t workspace_bytes, void* stream);
int kgc_shared_bwd_table(const int32_t* sorted_ids, const int32_t* sorted_slots, int32_t k, int64_t n_ent, int32_t D,
                         const float* d_rows, int64_t ld_rows, const float* d_row_bias, const float* scale, float* d_ent,
                         int64_t ld_d, float* d_bias, void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* KGC_B200_H_ */
