/*
 * lpformer_b200 — C ABI of the B200 (sm_100a) kernels behind LPFormer's per-link
 * pairwise-encoding path.
 *
 * The reference (HarryShomer/LPFormer) has no FFI: its hot path is Python calling
 * torch.sparse / torch_scatter / PyG library kernels.  Each entry point below names
 * the reference code it replaces (paths relative to the reference's src/).  The
 * Python module lpformer_b200.LinkTransformer binds these through ctypes with
 * tensor.data_ptr() values; nothing torch-typed crosses this boundary.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - no entry point allocates, synchronises or keeps global state (except the
 *     thread-local last-error string); launches are stream-ordered;
 *   - return value: 0 = success, negative = error (see lpf_last_error());
 *   - CSR tables: rowptr int64 [n+1], col int32 [nnz] ascending within a row,
 *     val fp32 [nnz];
 *   - links: int64 [2, BS] row-major (row 0 = source a, row 1 = target b), the
 *     layout of `batch` in models/link_transformer.py:82;
 *   - dense matrices are fp32 row-major with an explicit leading dimension.
 */
#ifndef LPFORMER_B200_H
#define LPFORMER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LPF_OK 0
#define LPF_ERR_INVALID -1   /* bad argument */
#define LPF_ERR_CUDA -2      /* CUDA runtime error (launch/config) */
#define LPF_ERR_UNSUPPORTED -3

/* selection modes, models/link_transformer.py:39-44 */
#define LPF_MODE_CN 0
#define LPF_MODE_1HOP 1
#define LPF_MODE_ALL 2

/* selection algorithms (same results, different work shapes):
 *   GENERIC    warp-per-link merge-path over both rows; valid for any thresholds / values.
 *   INTERSECT8 / INTERSECT32
 *              group-of-8 / warp-per-link walk of the shorter row with binary search into the
 *              longer one; links whose shorter row exceeds 16 elements per lane are deferred to a
 *              second launch in which a whole CTA walks each of them.  Requires th_1hop > 0 (modes 1HOP, ALL), th_non1hop > 0 (mode ALL) and
 *              every stored PPR value in (0, 1] (the caller asserts this for its table);
 *              otherwise LPF_ERR_UNSUPPORTED / undefined sets. */
#define LPF_ALGO_GENERIC 0
#define LPF_ALGO_INTERSECT8 1
#define LPF_ALGO_INTERSECT32 2
/* PACKED: one-pass selection over the packed link rows of lpf_pack_link_rows (lpf_select_onepass_packed only);
 *         same preconditions as the INTERSECT algorithms. */
#define LPF_ALGO_PACKED 3

/* node-set types, concatenation order of models/link_transformer.py:161 */
#define LPF_T_CN 0
#define LPF_T_1HOP 1
#define LPF_T_NON1HOP 2

/* GEMM epilogue flags */
#define LPF_EPI_NONE 0
#define LPF_EPI_RELU 1
#define LPF_EPI_SIGMOID 2

int lpf_abi_version(void);
/* Thread-local description of the last error returned on this thread. */
const char* lpf_last_error(void);
/* 1 if a CUDA device of compute capability 10.x is current, else 0 (no error set). */
int lpf_device_ok(void);

/* ------------------------------------------------------------------------- *
 * K1  node selection — replaces compute_node_mask / get_ppr_vals /
 *     get_non_1hop_ppr (models/link_transformer.py:214-319, :434-481) and the
 *     scatter counts of get_structure_cnts/get_count (:340-386).
 *
 * Pass 1 (count): counts[t*BS + i] = |set_t(link i)| for t in {CN,1HOP,NON1HOP}
 *                 (types the mode does not produce are written as 0).
 * Scan          : ptr[0..3*BS] = exclusive prefix sum of counts (int64), so type t
 *                 of link i owns rows [ptr[t*BS+i], ptr[t*BS+i+1]) of the pair
 *                 arrays; the pair arrays are therefore ordered type-major, then
 *                 by (link, node) — the order of torch.cat((cn, onehop, non1hop)).
 * Pass 2 (fill) : node[s], src_ppr[s], tgt_ppr[s] (and link[s] if non-NULL).
 * src_ppr/tgt_ppr are q(P(a,u)), q(P(b,u)) with q(p) = fl32(p+1)-1 (absent -> 0),
 * the value the reference thresholds and feeds to the RPE MLPs.
 * ------------------------------------------------------------------------- */
int lpf_select_count(const int64_t* links, int64_t bs,
                     const int64_t* adj_rowptr, const int32_t* adj_col,
                     const int64_t* ppr_rowptr, const int32_t* ppr_col, const float* ppr_val,
                     float th_cn, float th_1hop, float th_non1hop, int mode, int algo,
                     int32_t* counts, void* workspace, void* stream);

/* Bytes of device workspace the INTERSECT algorithms need for a batch of bs links (the count pass records
 * the links it defers to the CTA-wide kernel there; the fill pass of the SAME batch must get the same
 * buffer, untouched in between).  GENERIC ignores the workspace (may be NULL). */
int64_t lpf_select_workspace_bytes(int64_t bs);

/* Exclusive scan of n int32 counts into n+1 int64 offsets (single launch).
 * `scratch` must hold lpf_scan_scratch_bytes(n) bytes. */
int64_t lpf_scan_scratch_bytes(int64_t n);
int lpf_scan_counts(const int32_t* counts, int64_t n, int64_t* ptr, void* scratch, void* stream);

/* ------------------------------------------------------------------------- *
 * Device-side sizes.  Entry points with a trailing `const int64_t* *_dev` argument accept a DEVICE pointer to
 * the actual row / link count; the host-side count is then only the capacity the grid and the buffers were
 * sized for (actual = min(capacity, *dev)).  With them a whole batch runs without a host round trip and can be
 * captured in a CUDA graph.  Pass NULL for the plain host-sized behaviour.
 *
 * One-pass selection (INTERSECT algorithms only): counts, allocates and writes in a single launch sequence.
 * Pairs of type t go to rows [t*cap, t*cap + header[t]) of node / src_ppr / tgt_ppr (arrays of 3*cap rows);
 * within a type a link's pairs are contiguous and ascending, links appear in arbitrary order.  Outputs:
 * counts[t*BS+i], seg_start[t*BS+i] (first row relative to t*cap), nz_list (batch positions of the links with
 * a non-empty set), header int64[8] = (pairs of type 0, 1, 2, non-empty links, overflow flag, ...).  If a pool
 * overflows, header[4] = 1, header[0..3] = 0 and the pair arrays are undefined: re-run the batch through
 * count / scan / fill.
 * ------------------------------------------------------------------------- */
int lpf_select_onepass(const int64_t* links, int64_t bs,
                       const int64_t* adj_rowptr, const int32_t* adj_col,
                       const int64_t* ppr_rowptr, const int32_t* ppr_col, const float* ppr_val,
                       float th_cn, float th_1hop, float th_non1hop, int mode, int algo, int64_t cap,
                       int32_t* counts, int32_t* seg_start, int32_t* nz_list, int64_t* header,
                       int32_t* node, float* src_ppr, float* tgt_ppr, void* workspace, void* stream);

/* ------------------------------------------------------------------------- *
 * Packed link rows: the HBM layout of the per-link walk.  The reference slices rows a and b out of two N x N
 * sparse COO tensors with four index_select calls per batch (models/link_transformer.py:229-230, :290-291,
 * :444-449); the CSR tables above already make that a direct row access, but a link's target still costs four
 * dependent random reads in four arrays, and DRAM serves random reads in 128-byte lines whatever part of a line is
 * used (tools/gather_probe.cu).  lpf_pack_link_rows rewrites (adjacency CSR, PPR CSR) once per graph as
 *   slab     : one 128-byte line per node, node x at byte x * 128 (no locator): chunk 0 = header
 *              (uint32 deg, uint32 nP, uint32 first 128-byte unit of the row's overflow, 0), chunks 1..7 = the first
 *              seven 16-byte chunks of the row
 *   overflow : the remaining chunks of the rows longer than seven chunks, each row's part 128-byte aligned
 *   a row    = ceil(nP/2) PPR chunks — two entries (column | 0x80000000, value bits) in ascending column order, the
 *              odd one out padded with (0xffffffff, 0) — then ceil(deg/4) id chunks: four ascending neighbour ids,
 *              padded with 0x7fffffff
 * so that the median target is ONE line and one trip (link -> slab line) and the others one more.
 * slab needs lpf_link_rows_slab_bytes(n) bytes, overflow lpf_link_rows_bytes(n, adj_nnz, ppr_nnz) bytes (an upper
 * bound; -1 if the unit index would not fit 32 bits), both 128-byte aligned; scratch lpf_link_rows_scratch_bytes(n).
 *
 * lpf_select_onepass_packed is lpf_select_onepass (same outputs, same header protocol, same preconditions as
 * the INTERSECT algorithms) on those rows: one CTA per piece of 256 links (1-3 runs of equal source), four per SM.
 * The CTA stages the sources of its piece in shared memory (bucketed hash set of A(a), tables of P(a)) while the
 * slab lines of its targets are in flight; then every warp screens its own 32 links (slab line, then the overflow
 * chunks flattened into a list, one lane per chunk) and resolves the ones that select anything.  Rows of more
 * than 1,024 chunks go to the deferred-link kernel (walk of the short source row over the CSR tables); runs whose
 * source does not fit the table take a second launch with a larger one; the CSR tables are also read by the
 * fallbacks (pieces that are not runs of equal source, sources beyond even the larger table).
 * ------------------------------------------------------------------------- */
int64_t lpf_link_rows_slab_bytes(int64_t n);
int64_t lpf_link_rows_bytes(int64_t n, int64_t adj_nnz, int64_t ppr_nnz);
int64_t lpf_link_rows_scratch_bytes(int64_t n);
int lpf_pack_link_rows(const int64_t* adj_rowptr, const int32_t* adj_col,
                       const int64_t* ppr_rowptr, const int32_t* ppr_col, const float* ppr_val, int64_t n,
                       void* slab, void* overflow, void* scratch, void* stream);
int lpf_select_onepass_packed(const int64_t* links, int64_t bs,
                              const int64_t* adj_rowptr, const int32_t* adj_col,
                              const int64_t* ppr_rowptr, const int32_t* ppr_col, const float* ppr_val,
                              const void* slab, const void* overflow,
                              float th_cn, float th_1hop, float th_non1hop, int mode, int64_t cap,
                              int32_t* counts, int32_t* seg_start, int32_t* nz_list, int64_t* header,
                              int32_t* node, float* src_ppr, float* tgt_ppr, void* workspace, void* stream);

/* After the scan: batch positions of the links with at least one selected node (nz_list int32 [<= BS], any
 * order) and header int64[4] = (S_cn, S_cn + S_1hop, S, number of non-empty links) — the one small read-back
 * the host needs to size the pair arrays and the compacted attention batch. */
int lpf_select_compact(const int64_t* ptr, int64_t bs, int32_t* nz_list, int64_t* header, void* stream);

int lpf_select_fill(const int64_t* links, int64_t bs,
                    const int64_t* adj_rowptr, const int32_t* adj_col,
                    const int64_t* ppr_rowptr, const int32_t* ppr_col, const float* ppr_val,
                    float th_cn, float th_1hop, float th_non1hop, int mode, int algo,
                    const int64_t* ptr,
                    int32_t* node, float* src_ppr, float* tgt_ppr, int32_t* link /* may be NULL */,
                    void* workspace, void* stream);

/* ------------------------------------------------------------------------- *
 * RPE hidden vector — first half of get_pos_encodings (models/link_transformer.py
 * :182-211) with MLP = Linear(2,d) -> LayerNorm -> ReLU (models/other_models.py
 * :125-133):  hsum[s,:] = h(pa,pb) + h(pb,pa),  h(x,y) = ReLU(LN(W1 [x,y] + b1)).
 * The second Linear and lin_r's PE half are folded into one contraction done by
 * lpf_gemm (SURVEY App. B).  w1 is the [d,2] weight, b1/ln_w/ln_b are [d].
 * Rows [row0, row0+rows) of the pair arrays are processed (one type at a time).
 * ------------------------------------------------------------------------- */
int lpf_rpe_hidden(const float* src_ppr, const float* tgt_ppr, int64_t row0, int64_t rows,
                   const float* w1, const float* b1, const float* ln_w, const float* ln_b,
                   int32_t d, float* hsum, int64_t ld_hsum, const int64_t* rows_dev, void* stream);

/* ------------------------------------------------------------------------- *
 * Dense contraction  C[M,N] = epi( A[M,K] . W[N,K]^T + bias[N] )  — every
 * nn.Linear on the path (modules/layers.py:130-131,208-214; models/other_models.py
 * :125-138,173-179; GCNConv.lin).  W is the nn.Linear weight layout.  bias may be
 * NULL.  `bias_scale` multiplies the bias (2.0 for lin_l(e1)+lin_l(e2)).
 * ------------------------------------------------------------------------- */
int lpf_gemm(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias,
             float bias_scale, float* C, int64_t ldc, int64_t M, int32_t N, int32_t K,
             int epilogue, void* stream);

/* The same contraction on the tcgen05 tensor cores (kind::tf32 with the 3xTF32 split, fp32-level accuracy;
 * accumulators in TMEM, weights staged by bulk TMA copies).  `Wpacked` is the pre-split, pre-swizzled image of
 * the nn.Linear weight W[N,K] built once per weight by lpf_pack_weight into lpf_pack_weight_bytes(N,K) bytes
 * of device memory (16-byte aligned).  N <= 256 per call (split larger weights by rows). */
int64_t lpf_pack_weight_bytes(int32_t N, int32_t K);
int lpf_pack_weight(const float* W, int64_t ldw, int32_t N, int32_t K, float* packed, void* stream);
int lpf_gemm_tc(const float* A, int64_t lda, const float* Wpacked, const float* bias, float bias_scale,
                float* C, int64_t ldc, int64_t M, int32_t N, int32_t K, int epilogue, const int64_t* m_dev,
                void* stream);

/* Row-wise LayerNorm (eps 1e-5) over the first `n` columns, optional ReLU, in place
 * or out of place (X may equal Y).  nn.LayerNorm + F.relu of MLP/GCN/gnn_norm.
 * If `residual` is non-NULL the result is residual + act(LN(x)) (GCN.forward :71).
 * gamma == beta == NULL skips the normalisation (GCN with layer_norm=False). */
int lpf_layernorm_act(const float* X, int64_t ldx, const float* gamma, const float* beta,
                      const float* residual, int64_t ldr, float* Y, int64_t ldy,
                      int64_t rows, int32_t n, int relu, const int64_t* rows_dev, void* stream);

/* Link-level gathers (models/link_transformer.py:101-102,143-144; train/testing.py:29,113):
 * xsum[i,:] = X[a_i,:] + X[b_i,:]   (input of lin_l, since lin_l(e1)+lin_l(e2) = W_l(e1+e2)+2b)
 * xprod[i,:] = X[a_i,:] * X[b_i,:]  (input of elementwise_lin).  Either output may be NULL. */
int lpf_gather_links(const int64_t* links, int64_t bs, const int32_t* idx /* NULL or [n] batch positions */,
                     int64_t n, const float* X, int64_t ldx, int32_t d,
                     float* xsum, int64_t ld_sum, float* xprod, int64_t ld_prod, const int64_t* n_dev,
                     int x_bf16 /* X holds bf16 (ldx in elements) */, void* stream);

/* Query groups -> links (train/testing.py:14-27: source.repeat(K) x negative targets).  The grouped form holds one
 * source per query and K targets per query; its flat link index i = q*K + j is link (source[q], targets[q*K + j]).
 * Writes the flat range of n links that starts at position j0 (0 <= j0 < K) of its first query:
 *   links[i] = source[(j0 + i) / K],  links[ld + i] = targets[i]   for i < n,
 * so `source` points at the first query the range touches and `targets` at the range's first target.  Both arrays hold
 * int32 (id_bytes 4) or int64 (id_bytes 8) ids; links is int64 [2, ld] with ld >= n.  An id outside [0, num_nodes) is
 * written as 0 (no later kernel reads out of bounds) and sets *bad (int64) to non-zero; the caller resets *bad.
 * n == 0 is a no-op. */
int lpf_expand_query_links(const void* source, const void* targets, int32_t id_bytes, int64_t K, int64_t j0, int64_t n,
                           int64_t num_nodes, int64_t* links, int64_t ld, int64_t* bad, void* stream);

/* Source sweep -> links: every node in [0, n_targets) as a target of every source.  Flat link i = q*n_targets + j is
 * link (source[q], j).  Writes the flat range of n links that starts at position j0 (0 <= j0 < n_targets) of its first
 * query:  links[i] = source[(j0 + i) / n_targets],  links[ld + i] = (j0 + i) % n_targets   for i < n,
 * so `source` points at the first query the range touches.  source holds int32 (id_bytes 4) or int64 (id_bytes 8)
 * ids; n_targets <= num_nodes.  A source outside [0, num_nodes) is written as 0 and sets *bad (int64) to non-zero; the
 * caller resets *bad.  n == 0 is a no-op. */
int lpf_expand_source_sweep(const void* source, int32_t id_bytes, int64_t n_targets, int64_t j0, int64_t n,
                            int64_t num_nodes, int64_t* links, int64_t ld, int64_t* bad, void* stream);

/* Bytes of workspace lpf_topk_fold needs for a range of up to bs scores (-1 for bad arguments). */
int64_t lpf_topk_fold_workspace_bytes(int64_t bs, int32_t k, int64_t n_targets);

/* Folds the scores prob[0, n) of the flat sweep positions [lo, lo + n) (position q*n_targets + j: source[q], target j)
 * into per-query state, for num_queries queries:
 *   top_key fp32 [num_queries, k], top_id int32 [num_queries, k]: the k best candidates so far, ordered by (score
 *     descending, target id ascending); slots never filled hold (-inf, -1).  Initialise them so before the first fold.
 *   cnt_ge, cnt_gt int64 [num_queries] (with positives): candidates with score >= / > pos_score[q], accumulated.
 * The candidates of query q are all j in [0, n_targets) except source[q] and the ids of the exclusion row of source[q]
 * (ex_rowptr / ex_col: a CSR of ex_rows rows, col ascending within a row; NULL for none; a source outside [0, ex_rows)
 * has no row).  The counters also leave out positive[q].  source and positive are int32 or int64 (id_bytes), indexed
 * from query 0; positive, pos_score, cnt_ge and cnt_gt are all given or all NULL.  1 <= k <= 1024.
 * The state after any sequence of folds depends only on the multiset of (query, target, score) folded, not on how the
 * positions were cut into ranges or in which order the ranges came.
 * skip (NULL = never): when *skip is non-zero on the device at launch time, the call folds nothing (a batch whose
 * scores are invalid, e.g. a pair-pool overflow flag, can be folded later without a host round trip).
 * workspace: >= lpf_topk_fold_workspace_bytes(n, k, n_targets) bytes.  n == 0 is a no-op. */
int lpf_topk_fold(const float* prob, int64_t lo, int64_t n, const void* source, const void* positive, int32_t id_bytes,
                  int64_t num_queries, int64_t n_targets, const int64_t* ex_rowptr, const int32_t* ex_col,
                  int64_t ex_rows, const float* pos_score, int32_t k, float* top_key, int32_t* top_id, int64_t* cnt_ge,
                  int64_t* cnt_gt, const int64_t* skip, void* workspace, int64_t workspace_bytes, void* stream);

/* dst[r,:] = fill_row[:] for all `rows` rows (skipped when fill_row is NULL), then dst[idx[j],:] = src[j,:]
 * for j < n: puts the pairwise rows of the compacted non-empty links back in batch order, every other link
 * getting the constant empty-set row. */
int lpf_scatter_rows(const float* src, int64_t ld_src, const int32_t* idx, int64_t n,
                     float* dst, int64_t ld_dst, int64_t rows, int32_t d, const float* fill_row, void* stream);

/* ------------------------------------------------------------------------- *
 * K4  fused per-link attention — replaces LinkTransformerLayer.forward +
 * LinkAttention.forward/message (modules/layers.py:39-82,161-224): for link i and
 * each selected pair s (all three type segments):
 *     v_s   = KV[node[s],:] + R[s,:]                     (lin_r, split as in App. B)
 *     sc_sh = sum_c att[h,c] * leaky_relu(v_s[h,c] * Q[i,h,c], 0.2)
 *     alpha = segment softmax over the link's pairs (max-subtracted, denom + 1e-16)
 *     out_i = LayerNorm_{H*C}( sum_s alpha_s v_s + bias )
 * and appends the set counts (get_structure_cnts) as fp32 columns after the H*C
 * outputs: mode ALL -> (cn, 1hop, non1hop, cn+1hop); 1HOP -> (cn, 1hop, cn+1hop);
 * CN -> (cn); pass write_counts=0 for inner layers of a multi-layer stack.
 * alpha_out (may be NULL) receives the head-mean attention weight per pair.
 * With idx != NULL only the n listed links are processed and rows j of Q / out belong to link idx[j]
 * (the compacted list of lpf_select_compact); otherwise n == bs and row j is link j.
 * With seg_start != NULL (one-pass selection) type t of link i owns pair rows [t*type_stride + seg_start[t*bs+i],
 * + seg_cnt[t*bs+i]) and ptr is ignored.
 * ------------------------------------------------------------------------- */
int lpf_attend_fused(const int64_t* ptr, int64_t bs, const int32_t* idx /* NULL or [n] batch positions */,
                     int64_t n, const int32_t* node,
                     const float* KV, int64_t ld_kv, const float* R, int64_t ld_r,
                     const float* Q, int64_t ld_q,
                     const float* att, const float* bias, const float* ln_w, const float* ln_b,
                     int32_t heads, int32_t ch, int mode, int write_counts,
                     float* out, int64_t ld_out, float* alpha_out,
                     const int64_t* n_dev, const int32_t* seg_start, const int32_t* seg_cnt, int64_t type_stride, int kv_bf16 /* KV holds bf16 (ld_kv in elements) */,
                     void* stream);
/* The same with a caller-owned DEVICE workspace (16-byte aligned, at least lpf_attend_workspace_min() bytes, no
 * initialisation needed, private to the call's stream while it runs): a link with more than 1,024 selected pairs (dense
 * graphs: two hubs of the ogbl-ppa shape share tens of thousands of common neighbours) is then left out of the first
 * launch, registered in the workspace, and walked in a second launch by many CTAs at once, 256 pairs each — partial
 * softmax states (running max, denominator, weighted sum) go to the workspace and the CTA that completes a link's
 * last chunk merges them.  Same results up to fp32 re-association of the softmax sums.  Links that do not fit the
 * workspace (1,024 links, (bytes - 16 KB) / (4 (2 H + 32 H ceil(C/32))) chunk records) are walked by their own CTA
 * as without a workspace.
 * r_map / r_const: pairs whose two (quantised) PPR values are 0 — most common neighbours of a dense graph under
 * thresh_cn = 0 have no PPR entry — share ONE relative-positional-encoding row per node type (the RPE MLP sees (0, 0),
 * models/link_transformer.py:182-211); with a row map the caller computes R only for the other pairs (compacted) and the
 * kernel reads the per-type constant row for the rest. */
int64_t lpf_attend_workspace_min(void);
int lpf_attend_fused_ws(const int64_t* ptr, int64_t bs, const int32_t* idx, int64_t n, const int32_t* node,
                        const float* KV, int64_t ld_kv, const float* R, int64_t ld_r,
                        const float* Q, int64_t ld_q,
                        const float* att, const float* bias, const float* ln_w, const float* ln_b,
                        int32_t heads, int32_t ch, int mode, int write_counts,
                        float* out, int64_t ld_out, float* alpha_out,
                        const int64_t* n_dev, const int32_t* seg_start, const int32_t* seg_cnt, int64_t type_stride, int kv_bf16,
                        const int32_t* r_map /* NULL, or [S]: pair s reads R[r_map[s]] if >= 0, else r_const[-1 - r_map[s]] */,
                        const float* r_const /* [3, ld_r]: the RPE row of a pair with two zero PPR values, per node type */,
                        void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------- *
 * Fused per-link heads on the tensor cores (d in {32, 64}) — the rest of the eval-loop body
 * (train/testing.py:29-31,113-115) for links whose pairwise vector pw is known:
 *     prob = mlp_score([ elementwise_lin(X[a]*X[b]) | pw ])          (models/other_models.py:125-138,173-179)
 * with elementwise_lin = Linear(W1,b1) -> LayerNorm -> ReLU -> Linear(W2,b2) and mlp_score = Linear(Ws1,bs1) ->
 * ReLU -> Linear(ws2,bs2) -> sigmoid.  W2 and Ws1[:, :d] are adjacent linear maps and are folded by the caller:
 *     w23 = Ws1[:, :d] W2  [2d, d],   offset = Ws1[:, :d] b2 + bs1 + Ws1[:, d:] pw  [2d]
 *     prob = sigmoid(ws2 . ReLU(w23 ReLU(LN(W1 (X[a]*X[b]) + b1)) + offset) + bs2).
 * offset is either the constant c3 (links whose selected sets are all empty share one pw) or per-row zb [n, 2d].
 * w1_packed / w23_packed are lpf_pack_weight images.  idx (optional) lists the batch positions to score;
 * prob[pos] is written (the pre-sigmoid logit when logits != 0).
 * tile_sched (optional): two zero-initialised int32 words owned by the caller, {next tile, finished CTAs}.  With
 * it the CTAs of the launch take their 128-link tiles from a counter instead of a fixed stride (a CTA that starts
 * late, because its SM was still busy with another stream's kernel, then simply takes fewer tiles); the last CTA
 * to finish re-arms the words, so one pair serves every launch on a stream.
 * ------------------------------------------------------------------------- */
int lpf_link_heads_tc(const int64_t* links, int64_t bs, const int32_t* idx, int64_t n,
                      const float* X, int64_t ldx, int32_t d,
                      const float* w1_packed, const float* b1, const float* ln_w, const float* ln_b,
                      const float* w23_packed, const float* c3, const float* zb, int64_t ld_zb,
                      const float* ws2, const float* bs2, float* prob, int logits, const int64_t* n_dev,
                      int32_t* tile_sched, void* stream);

/* ------------------------------------------------------------------------- *
 * The same head chain with fp16-split operands (d = 64): tcgen05.mma.kind::f16 on x = hi + lo, hi = fp16(x s),
 * lo = fp16(x s - hi) — the 22 significand bits of the 3xTF32 split at half the tensor-pipe time and half the
 * operand bytes.  s is an exact power of two per operand, undone in the epilogues:
 *   * w1_packed / w23_packed: lpf_pack_weight_f16 images built with a scale that puts max|W| into [2^14, 2^15);
 *     inv_scale_w1 = 1 / scale(W1), inv_scale_h_w23 = 1 / (s_h scale(W23));
 *   * ln_w_scaled / ln_b_scaled: LayerNorm weight and bias times s_h, s_h a power of two with
 *     s_h (sqrt(d) max|ln_w| + max|ln_b|) <= 2^15 (LayerNorm bounds h, so h s_h fits fp16);
 *   * the gathered rows X[a]*X[b] are scaled per link inside the kernel.
 * The X[b] rows are fetched by TMA row gathers (tile::gather4) through a tensor map of X [n_nodes, d] built per call:
 * X rows must be 16-byte aligned, and every link id must be < n_nodes.  x_bf16 != 0: X holds bf16 (the node table at
 * half the bytes; ldx in elements; arithmetic unchanged: fp32 products, fp16-split contractions, fp32 accumulation).
 * Everything else as lpf_link_heads_tc (no tile_sched).
 * ------------------------------------------------------------------------- */
int64_t lpf_pack_weight_f16_bytes(int32_t N, int32_t K);
int lpf_pack_weight_f16(const float* W, int64_t ldw, int32_t N, int32_t K, float scale, void* packed, void* stream);
int lpf_link_heads_f16(const int64_t* links, int64_t bs, const int32_t* idx, int64_t n,
                       const void* X, int x_bf16, int64_t ldx, int64_t n_nodes, int32_t d,
                       const void* w1_packed, float inv_scale_w1, const float* b1,
                       const float* ln_w_scaled, const float* ln_b_scaled,
                       const void* w23_packed, float inv_scale_h_w23, const float* c3, const float* zb, int64_t ld_zb,
                       const float* ws2, const float* bs2, float* prob, int logits, const int64_t* n_dev,
                       void* stream);
/* Profiling hook of lpf_link_heads_f16 (as lpf_debug_heads_clocks). */
int lpf_debug_heads_f16_clocks(void* device_buffer);

/* ------------------------------------------------------------------------- *
 * Fused path for links with a non-empty node set, small-batch regime: one warp takes one link of nz_list
 * (n = min(n_cap, *n_dev)) from its node sets (one-pass selection buffers) to its score — lin_l, the RPE MLP and
 * its contraction per pair, attention with online segment softmax, bias + LayerNorm + counts, pairwise_lin,
 * elementwise_lin and mlp_score — in fp32 FFMA, replacing lpf_gather_links / lpf_rpe_hidden / lpf_gemm_tc x7 /
 * lpf_attend_fused / lpf_layernorm_act / lpf_link_heads_tc on the compacted list when that list is a few
 * thousand links (where those launches are latency, not work).  d in {32, 64}, heads = 1, one attention layer.
 * Every `*T` matrix is the TRANSPOSE of the nn.Linear weight (row k = input channel k, contiguous outputs):
 *   wlT = lin_l.weight^T [d][d];  rpe_mT[t] = (W_pe W2_t)^T [d][d], rpe_c[t] = 2 W_pe b2_t + b_r (SURVEY App. B);
 *   p1T / p2T = pairwise_lin.linears.{0,1}.weight^T [pd][pd] / [pd][d], pd = d + count_dim;
 *   wzT = Ws1[:, d:]^T [d][2d], off = Ws1[:, :d] b2 + bs1;  w1T = elementwise_lin.linears.0.weight^T [d][d];
 *   w23T = (Ws1[:, :d] W2)^T [d][2d]  (the folding of lpf_link_heads_tc).
 * ------------------------------------------------------------------------- */
typedef struct lpf_nz_args {
    const int64_t* links; int64_t bs;
    const int32_t* nz; int64_t n_cap; const int64_t* n_dev;
    const float* X; int64_t ldx;
    const float* KV; int64_t ld_kv;
    const int32_t* node; const float* src_ppr; const float* tgt_ppr;
    const int32_t* seg_start; const int32_t* counts; int64_t cap;
    const int64_t* header;   /* one-pass selection header: [0..2] pairs per type */
    float* R;                /* scratch [3*cap, d]: RPE contraction per pair */
    int32_t d; int32_t mode;
    const float* wlT; const float* bl;
    const float* rpe_w1[3]; const float* rpe_b1[3]; const float* rpe_ln_w[3]; const float* rpe_ln_b[3];
    const float* rpe_mT[3]; const float* rpe_c[3];
    const float* att; const float* att_bias; const float* post_ln_w; const float* post_ln_b;
    const float* p1T; const float* pb1; const float* pln_w; const float* pln_b; const float* p2T; const float* pb2;
    const float* wzT; const float* off;
    const float* w1T; const float* b1; const float* ln_w; const float* ln_b;
    const float* w23T; const float* ws2; const float* bs2;
    float* prob; int32_t logits;
    int32_t tab_bf16;   /* X and KV hold bf16 (leading dimensions in elements) */
} lpf_nz_args;
int lpf_nz_links_fused(const lpf_nz_args* args, void* stream);
/* The pair stage of lpf_nz_links_fused alone: R[t * cap + r] = (h(pa,pb) + h(pb,pa)) (W_pe W2_t)^T + c_t for the
 * header[t] selected pairs of every type t (models/link_transformer.py:182-211) in ONE launch — what three
 * lpf_rpe_hidden + three lpf_gemm_tc launches compute in the batched regime.  Reads of `args`: src_ppr, tgt_ppr, cap,
 * header, R, d, mode and the rpe_* parameters. */
int lpf_nz_pairs(const lpf_nz_args* args, void* stream);

/* Profiling hook: later lpf_select_onepass_packed launches add per-phase clock64() totals of the screening kernel into
 * device_buffer (int64[48]: [0] source staging, [1] phase A, [2] phase B, [3] phase C, [4] generic fallback,
 * [5] pieces, [6] links resolved by a warp, [7] by the whole CTA, [8..9] slowest piece / CTA, [10..13] set-up phases,
 * [16..38] the slowest piece's own phases and sizes; see tools/select_clocks.py); NULL disables. */
int lpf_debug_select_clocks(void* device_buffer);

/* Profiling hook: with enable != 0 later lpf_select_onepass_packed calls record CUDA events on their stream around
 * the screening kernel, the resolve kernel, the hub-hub resolve kernel and the deferred-link tail;
 * lpf_debug_select_timing_read waits for the last such call and stores the four durations (milliseconds) in
 * ms4_host[0..3]; -1 if nothing was recorded. */
int lpf_debug_select_timing(int enable);
int lpf_debug_select_timing_read(float* ms4_host);
/* Test hook: caps the hash slots lpf_select_onepass_packed's screening launch may use for the staged sources (its
 * hub launch gets four times as many), so that small graphs reach the hub launch and the global-memory search of
 * sources beyond it; 0 restores the full tables. */
int lpf_debug_select_slots(int limit);
/* Same switch: the two kernels of the last lpf_nz_links_fused call (pair stage, link stage) in ms2_host[0..1]. */
int lpf_debug_nz_timing_read(float* ms2_host);

/* Profiling hook: CTA 0 of later lpf_link_heads_tc launches writes clock64() stamps of its pipeline phases for
 * its first 8 tiles into device_buffer (int64 [8][16]); NULL disables. */
int lpf_debug_heads_clocks(void* device_buffer);

/* ------------------------------------------------------------------------- *
 * K2  GCN message passing — GCNConv's SpMM (models/other_models.py:66 via
 * torch_sparse.matmul): Y[r,:] = sum_k val[k] * XW[col[k],:] + bias over CSR row r,
 * for rows [row0, row0+rows) (row sharding for multi-GPU).
 * ------------------------------------------------------------------------- */
int lpf_gcn_spmm(const int64_t* rowptr, const int32_t* col, const float* val,
                 int64_t row0, int64_t rows, const float* XW, int64_t ld_xw, const float* bias,
                 int32_t d, float* Y, int64_t ldy, void* stream);
/* The same SpMM with the rest of the GCN layer fused into its epilogue (GCN.forward, models/other_models.py:66-72,
 * and for the last layer LinkTransformer.gnn_norm, models/link_transformer.py:126):
 *     Y[r,:] = LN2( residual[r,:] + act( LN1( sum_k val[k] XW[col[k],:] + bias ) ) )
 * ln_w/ln_b (LN1), relu, residual (rows indexed like Y), ln2_w/ln2_b (LN2) are each optional (NULL / 0).  Needs
 * d % 4 == 0, d <= 512 and 16-byte aligned rows / vectors (LPF_ERR_UNSUPPORTED otherwise: use lpf_gcn_spmm +
 * lpf_layernorm_act). */
int lpf_gcn_layer(const int64_t* rowptr, const int32_t* col, const float* val,
                  int64_t row0, int64_t rows, const float* XW, int64_t ld_xw, const float* bias, int32_t d,
                  const float* ln_w, const float* ln_b, int relu, const float* residual, int64_t ld_res,
                  const float* ln2_w, const float* ln2_b, float* Y, int64_t ldy, void* stream);

/* ------------------------------------------------------------------------- *
 * Host-side PPR precompute (data preparation, not on the per-link path) — the
 * Andersen push of util/calc_ppr_scores.py:137-192 + the fp32 sorted matrix of
 * :221-241, multi-threaded over sources, bit-identical values.  HOST pointers.
 * lpf_ppr_push_host returns an opaque handle (NULL on error) and the entry count;
 * lpf_ppr_push_host_fetch copies the CSR out (rowptr [n+1], col/val [nnz]) and
 * releases the handle.
 * ------------------------------------------------------------------------- */
/* ------------------------------------------------------------------------- *
 * PPR precompute on the GPU (SURVEY 8(f) rank 1): the same push (util/calc_ppr_scores.py:137-192), one warp per
 * source, bit-identical values (tests compare with lpf_ppr_push_host).  DEVICE pointers.
 *   lpf_ppr_push_slots(alpha, eps): hash slots per warp = power of two >= 2 (1 + 1 / (alpha eps)), -1 if that is
 *     beyond 2^24 (use the host tool for such eps);  lpf_ppr_push_scratch_bytes(slots, nwarps): scratch size.
 *   lpf_ppr_push: sources [src0, src0 + nsrc) — or src_list[0 .. nsrc) when src_list is given — of the CSR graph
 *     (sorted columns, no self loops) with `nwarps` resident warps (a multiple of 4) and `slots` hash slots each (any
 *     power of two >= 64: a source whose table fills up is skipped, counted in status[1] and listed in ovf_list if
 *     given, to be re-run with more slots); entries (row, col, fp32 value) are appended to the pool out_* [cap] through
 *     cursor[0] (int64, not reset: several source ranges can share a pool; cursor[1] is the work counter and must be 0
 *     on entry), in arbitrary order — sort by (row, col) for the CSR.  status[0] != 0: the pool was too small (the
 *     entries that did not fit are lost: retry with a larger cap); status[1]: number of sources whose table filled up
 *     (0 with slots = lpf_ppr_push_slots(alpha, eps) on a simple graph).
 * ------------------------------------------------------------------------- */
int32_t lpf_ppr_push_slots(double alpha, double eps);
int64_t lpf_ppr_push_scratch_bytes(int32_t slots, int32_t nwarps);
int lpf_ppr_push(const int64_t* indptr, const int32_t* indices, int64_t n, double alpha, double eps,
                 int64_t src0, int64_t nsrc, const int32_t* src_list, int32_t* ovf_list,
                 int32_t slots, int32_t nwarps, void* scratch,
                 int32_t* out_row, int32_t* out_col, float* out_val, int64_t cap, int64_t* cursor,
                 int32_t* status, void* stream);

void* lpf_ppr_push_host(const int64_t* indptr_host, const int32_t* indices_host, int64_t n,
                        double alpha, double eps, int nthreads, int64_t* nnz);
int lpf_ppr_push_host_fetch(void* handle, int64_t* rowptr_host, int32_t* col_host, float* val_host);

/* ------------------------------------------------------------------------- *
 * Backward pass (training, dropout included: see "Dropout" below): the gradients of the host-sized forward with respect to the reference's
 * parameters and to X_node.  Parameter gradients are reduced deterministically through a caller-owned workspace
 * (size from the matching *_workspace_bytes; -1 = bad arguments); `accumulate` != 0 adds into the outputs instead of
 * overwriting them.  Scatters into node-indexed tables (dX, dKV) are fp32 atomic adds into zero-initialised tables.
 *
 * lpf_layernorm_act_backward: y = act(LN(x)) of lpf_layernorm_act (nn.LayerNorm + F.relu of MLP, post_att_norm, the GCN's
 *   lns / gnn_norm; models/other_models.py:66-72,125-133, modules/layers.py:80) from the saved pre-norm rows x:
 *   dX (+)= dx, dgamma / dbeta (+)= column sums.  gamma == beta == NULL: ReLU (or identity) only.  n <= 1024.
 * lpf_gemm_wgrad: dW[N,K] (+)= dY[M,N]^T A[M,K] and db[N] (+)= sum of dY's rows, for nn.Linear / GCNConv.lin /
 *   lin_l / lin_r / the RPE contraction over M links, pairs or nodes (rows split over the grid, fp32 FFMA).  dW or db
 *   may be NULL (A may be NULL when dW is).  dX = dY W goes through lpf_gemm_tc on the transposed weight.
 * lpf_act_backward: dX = dY [Y > 0] (act = LPF_EPI_RELU) or dY Y (1 - Y) (LPF_EPI_SIGMOID) from the saved output Y
 *   (MLP without norm, mlp_score; models/other_models.py:173-179).
 * lpf_gather_links_backward: the transpose of lpf_gather_links (X[a] * X[b] of elementwise_lin, X[a] + X[b] into lin_l;
 *   models/link_transformer.py:100-101, modules/layers.py:208-214): dX[a] += dsum + dprod X[b], dX[b] += dsum + dprod X[a].
 * lpf_scatter_rows_backward: the transpose of lpf_scatter_rows with a fill row: dsrc[j] = dG[idx[j]] (dsrc may be NULL)
 *   and dfill = the sum of the rows of dG that idx does not name (the shared pairwise row of the links with empty sets).
 * lpf_rpe_hidden_backward: the first Linear + LayerNorm + ReLU of a PPR encoder (get_pos_encodings,
 *   models/link_transformer.py:182-211), both orderings (pa, pb) and (pb, pa), from dh = d hsum of rows
 *   [row0, row0 + rows) (dh row r belongs to pair row0 + r): dw1 [d, 2], db1, dln_w, dln_b.  d <= 256.
 * lpf_attend_backward: the segment-softmax attention of lpf_attend_fused_ws (modules/layers.py:39-82, :161-224) for the
 *   links of the batch (or the positions in idx), one warp per link at any set size, with its row map (r_map / r_const).
 *   From dY (the gradient of the layer's output rows, first heads*ch columns) it writes dQ [n, heads*ch], dR per pair row
 *   (rows the map names; every other pair's gradient is added into dR_const [3, heads*ch] by type), adds into dKV [N,
 *   heads*ch] and writes link_rows [n, 4 heads*ch] = (d o | dY LN-normalised o | dY | d att) per link, whose column
 *   sums (lpf_gemm_wgrad with dW = NULL) are the gradients of bias, post_att_norm.weight, post_att_norm.bias and att.
 * ------------------------------------------------------------------------- */
int64_t lpf_layernorm_act_backward_workspace_bytes(int64_t rows, int32_t n);
int lpf_layernorm_act_backward(const float* X, int64_t ldx, const float* gamma, const float* beta, int relu,
                               const float* dY, int64_t lddy, float* dX, int64_t lddx, int accumulate_dx,
                               float* dgamma, float* dbeta, int accumulate_param, int64_t rows, int32_t n,
                               void* workspace, int64_t workspace_bytes, void* stream);
int64_t lpf_gemm_wgrad_workspace_bytes(int64_t M, int32_t N, int32_t K);
int lpf_gemm_wgrad(const float* A, int64_t lda, const float* dY, int64_t lddy, int64_t M, int32_t N, int32_t K,
                   float* dW, int64_t ldw, float* db, int accumulate, void* workspace, int64_t workspace_bytes,
                   void* stream);
int lpf_act_backward(const float* Y, int64_t ldy, const float* dY, int64_t lddy, float* dX, int64_t lddx,
                     int64_t rows, int32_t n, int act, void* stream);
int lpf_gather_links_backward(const int64_t* links, int64_t bs, const int32_t* idx, int64_t n, const float* X,
                              int64_t ldx, int32_t d, const float* dsum, int64_t ld_sum, const float* dprod,
                              int64_t ld_prod, float* dX, int64_t lddx, void* stream);
int64_t lpf_scatter_rows_backward_workspace_bytes(int64_t rows, int32_t d);
int lpf_scatter_rows_backward(const float* dG, int64_t ldg, int64_t rows, int32_t d, const int32_t* idx, int64_t n,
                              float* dsrc, int64_t ld_src, float* dfill, void* workspace, int64_t workspace_bytes,
                              void* stream);
int64_t lpf_rpe_hidden_backward_workspace_bytes(int64_t rows, int32_t d);
int lpf_rpe_hidden_backward(const float* src_ppr, const float* tgt_ppr, int64_t row0, int64_t rows,
                            const float* w1, const float* b1, const float* ln_w, const float* ln_b, int32_t d,
                            const float* dh, int64_t ld_dh, float* dw1, float* db1, float* dln_w, float* dln_b,
                            int accumulate, void* workspace, int64_t workspace_bytes, void* stream);
int lpf_attend_backward(const int64_t* ptr, int64_t bs, const int32_t* idx, int64_t n, const int32_t* node,
                        const float* KV, int64_t ld_kv, const float* R, int64_t ld_r, const int32_t* r_map,
                        const float* r_const, const float* Q, int64_t ld_q, const float* att, const float* bias,
                        const float* ln_w, const float* ln_b, int32_t heads, int32_t ch, const float* dY,
                        int64_t ld_dy, float* dR, int64_t ld_dr, float* dR_const, float* dQ, int64_t ld_dq,
                        float* dKV, int64_t ld_dkv, float* link_rows, void* stream);

/* ------------------------------------------------------------------------- *
 * Dropout (training mode; F.dropout semantics: each element is zeroed with probability p, kept elements are scaled
 * by 1 / (1 - p); p outside [0, 1] is LPF_ERR_INVALID).  The sites and their `site` numbers (lpformer_b200/ops.py):
 * the GCN input features (1), node dropout of the selected pairs (2), GCN layer l (16 + l, after the activation),
 * attention layer l's output (32 + l), hidden layer i of an MLP / mlp_score (48 + i).
 *
 * Random numbers: counter-based Philox4x32-10 with key = the 64-bit seed (low word, high word) and counter =
 * (col >> 2, row low word, row high word, site); element (row, col) reads word col & 3.  `row` is the global row (the
 * node id of node tables, the batch position of link tables, the pair index of node dropout), so a mask does not depend
 * on row sharding (row0), index subsets or the launch shape.  Keep rule: the word u keeps the element iff
 * u >= floor(p 2^32); a kept element becomes x * fp32(1 / (1 - p)) (exactly that product), a dropped one 0.
 * The seed is read from device memory (`seed`: one uint64), so a seed drawn on the device needs no host sync.  Masks
 * are never stored: the backward regenerates them from the seed.
 *
 * lpf_dropout: Y[r, :n] = X[r, :n] * mask(row0 + r) / (1 - p) for rows [0, rows); X == Y is allowed (in place).  The
 *   forward of the feature, attention-output and MLP sites, the backward of every site (on dY), and on a table of ones
 *   the mask itself (mask / (1 - p)).
 * lpf_gcn_layer_dropout: lpf_gcn_layer with dropout between the activation and the residual:
 *   Y = LN2(residual + drop(act(LN1(A_hat XW + bias)))), mask row = node id.  (The reference's order conv -> LN ->
 *   dropout -> ReLU gives the same values: relu(m z / (1 - p)) == m relu(z) / (1 - p) exactly in fp32.)
 * lpf_layernorm_act_dropout: Y = residual + drop(act(LN(X))) (lpf_layernorm_act with the same dropout; mask row =
 *   row0 + r): the GCN backward's recompute of the rows that enter gnn_norm.
 * lpf_drop_pairs_count / lpf_drop_pairs_fill: node dropout (reference compute_node_mask -> drop_pairwise) of a
 *   selection (ptr [3 bs + 1], node / src_ppr / tgt_ppr / link [S], type-major, (link, node)-sorted): keeps exactly K
 *   pairs, a uniform K-subset (pair i's key: 64 Philox bits of (seed, site, row i, col 0) with its low
 *   ceil(log2 S) bits replaced by i; the K smallest keys are kept).  _count writes the kept pairs per (type, link)
 *   segment into counts [3 bs] (scan them with lpf_scan_counts into ptr_out, and lpf_select_compact gives the non-empty
 *   links and the new type bounds); _fill copies the kept pairs in order to ptr_out's positions (link / link_out may
 *   both be NULL).  The workspace (lpf_drop_pairs_workspace_bytes) carries the threshold from _count to _fill.
 * ------------------------------------------------------------------------- */
int lpf_dropout(const float* X, int64_t ldx, float* Y, int64_t ldy, int64_t rows, int32_t n, int64_t row0,
                const uint64_t* seed, int32_t site, double p, void* stream);
int lpf_gcn_layer_dropout(const int64_t* rowptr, const int32_t* col, const float* val, int64_t row0, int64_t rows,
                          const float* XW, int64_t ld_xw, const float* bias, int32_t d, const float* ln_w,
                          const float* ln_b, int relu, const uint64_t* seed, int32_t site, double p,
                          const float* residual, int64_t ld_res, const float* ln2_w, const float* ln2_b, float* Y,
                          int64_t ldy, void* stream);
int lpf_layernorm_act_dropout(const float* X, int64_t ldx, const float* gamma, const float* beta, int relu,
                              int64_t row0, const uint64_t* seed, int32_t site, double p, const float* residual,
                              int64_t ldr, float* Y, int64_t ldy, int64_t rows, int32_t n, void* stream);
int64_t lpf_drop_pairs_workspace_bytes(void);
int lpf_drop_pairs_count(const int64_t* ptr, int64_t bs, int64_t S, int64_t K, const uint64_t* seed, int32_t site,
                         int32_t* counts, void* workspace, int64_t workspace_bytes, void* stream);
int lpf_drop_pairs_fill(const int64_t* ptr, int64_t bs, const int32_t* node, const float* src_ppr,
                        const float* tgt_ppr, const int32_t* link, int64_t S, const uint64_t* seed, int32_t site,
                        const void* workspace, const int64_t* ptr_out, int32_t* node_out, float* src_out,
                        float* tgt_out, int32_t* link_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LPFORMER_B200_H */
