/*
 * eps.h — C ABI of libeps_b200.so: the B200 (sm_100a) kernels behind the
 * Edge-Proposal-Sets filter-and-rank scoring path.
 *
 * The reference (CUAI/Edge-Proposal-Sets) is pure Python and has no FFI of its
 * own; the boundary this library sits behind is the set of Python call sites
 * below (SURVEY.md §8b).  Each entry point cites the reference code it
 * replaces.  INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in _h;
 *   - `stream` is a CUstream / cudaStream_t passed as void* (NULL = default
 *     stream); all work is stream-ordered, no entry point synchronises;
 *   - the library never allocates device memory: outputs and workspaces are
 *     caller-owned, sizes come from the *_workspace_bytes functions;
 *   - node / neighbour indices are int32, CSR columns ascending inside a row,
 *     no duplicate entries (what rank.add_edges produces after to_symmetric);
 *   - return value: EPS_OK (0) or a negative eps_status; the message of the
 *     last failure on the calling thread is eps_last_error();
 *   - no CPU fallback exists: without a CUDA device every compute entry point
 *     returns EPS_ERR_CUDA.
 */
#ifndef EPS_B200_H
#define EPS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EPS_VERSION 203 /* 0.2.3; edge_proposal_sets_b200/_lib.py checks it at load time */

typedef enum {
  EPS_OK = 0,
  EPS_ERR_INVALID = -1,     /* bad argument (null pointer, negative size, k > M, ...) */
  EPS_ERR_CUDA = -2,        /* a CUDA runtime call or kernel launch failed */
  EPS_ERR_WORKSPACE = -3,   /* workspace too small */
  EPS_ERR_UNSUPPORTED = -4, /* shape outside what the kernel is built for */
  EPS_ERR_NCCL = -5
} eps_status;

int eps_version(void);
const char *eps_last_error(void);

/* ---------------------------------------------------------------------------
 * K1  CSR SpMM   Y = reduce_j( val_ij * X[col_j,:] ) (+ bias) (ReLU)
 * replaces: torch_sparse matmul(adj_t, x, reduce='add') inside GCNConv
 *           (/root/reference/models.py:183,186) and
 *           matmul(adj_t.set_value(None), x, reduce='mean') inside SAGEConv
 *           (/root/reference/models.py:436,439).
 * One warp per row, neighbours folded left-to-right in ascending column order
 * with fmaf (the accumulation order of torch_sparse's spmm kernel).
 *   val  == NULL : all ones.        reduce: EPS_REDUCE_SUM | EPS_REDUCE_MEAN
 *   bias == NULL : none.            relu  : 0 | 1 (applied after bias)
 * X and Y are row-major [n_cols_of_A, F] / [n_rows, F] fp32 and must not alias.
 * ------------------------------------------------------------------------- */
#define EPS_REDUCE_SUM 0
#define EPS_REDUCE_MEAN 1
int eps_spmm_csr_f32(const int32_t *rowptr, const int32_t *col, const float *val,
                     const float *X, float *Y, int32_t n_rows, int32_t F, int reduce,
                     const float *bias, int relu, void *workspace, size_t workspace_bytes,
                     void *stream);
size_t eps_spmm_workspace_bytes(void);

/* ---------------------------------------------------------------------------
 * K1b  GCN normalisation  A_hat = D^-1/2 (A with diag := 1) D^-1/2
 * replaces: torch_geometric gcn_norm inside GCNConv.forward, recomputed on every
 *           forward by the reference (cached=False, /root/reference/models.py:169-173,183,186).
 *   count: dinv[i] = (1 + sum_{j != i} w_ij)^-1/2 (inf -> 0); newlen[i] = row length with the
 *          diagonal entry present
 *   fill : rowptr2 = exclusive prefix sum of newlen (n+1 entries, caller computes it);
 *          col2 / val2 = columns with the diagonal merged in sorted position and
 *          val = (w * dinv[row]) * dinv[col]  (two fp32 roundings, that order)
 * ------------------------------------------------------------------------- */
int eps_gcn_norm_count(const int32_t *rowptr, const int32_t *col, const float *val, int32_t n,
                       float *dinv, int32_t *newlen, void *stream);
int eps_gcn_norm_fill(const int32_t *rowptr, const int32_t *col, const float *val, int32_t n,
                      const float *dinv, const int32_t *rowptr2, int32_t *col2, float *val2,
                      void *stream);

/* ---------------------------------------------------------------------------
 * K3  Common-Neighbour / Adamic-Adar / Resource-Allocation pair scores
 * replaces: CommonNeighborsPredictor.forward 'simple' and 'adamic'
 *           (/root/reference/models.py:536-554), adamic_utils.AA
 *           (/root/reference/adamic_utils.py:13-25) and
 *           train_and_eval.resource_allocation
 *           (/root/reference/train_and_eval.py:195-216).
 *   score[i] = RN_fp32( sum_{k in N(u_i) & N(v_i)} t_k ),  t_k = a_u * (a_v * w_k) in fp32;
 *              the t_k are added EXACTLY (64-bit fixed point, 38 fractional bits: exact for
 *              |t_k| >= 2^-15, <= 2^-39 absolute error per smaller term; |sum| < 2^25), so a
 *              score depends on (graph, u, v) only - not on order, batch, grid or GPU count
 *     a_u = val[u,k], a_v = val[v,k]  (1 when val == NULL)
 *     w_k = wtable[k]                 (1 when wtable == NULL -> plain CN)
 *   count[i] = |N(u_i) & N(v_i)|  (int32, exact)
 *   flags: EPS_CN_SIGMOID        apply 1/(1+exp(-x)) to score (models.py:554)
 *          EPS_CN_GROUPED_BY_V   promise: equal pair_v values come in long runs
 *                                (the column-major candidate order of
 *                                filter.py:96-109); selects the per-owner
 *                                shared-memory bitmap kernel.  Results are
 *                                identical with or without the flag.
 * score or count may be NULL (not both).
 * ------------------------------------------------------------------------- */
#define EPS_CN_SIGMOID 1
#define EPS_CN_GROUPED_BY_V 2
/* Degree-normalised similarity scores (eps_cn_aa, eps_twohop_onepass): a 3-bit kind field at
 * bit 8 of `flags`.  With c = |N(u) & N(v)| (the exact count), a = |N(u)|, b = |N(v)| (stored lists, self loops
 * included, edge values ignored), score =
 *   JACCARD        __fdiv_rn(c, a + b - c)             SORENSEN       __fdiv_rn(2c, a + b)
 *   HUB_PROMOTED   __fdiv_rn(c, min(a, b))             HUB_DEPRESSED  __fdiv_rn(c, max(a, b))
 *   SALTON         (float)((double)c / sqrt((double)a * (double)b))
 *   LHN            (float)((double)c / ((double)a * (double)b))      (Leicht-Holme-Newman)
 *   PREF_ATTACH    __ll2float_rn((int64)a * b)                         (preferential attachment)
 * A zero denominator gives 0.  The four divisions are correctly rounded when 2 * max degree < 2^24 (the caller
 * checks it).  A kind needs wtable == NULL, val == NULL and no EPS_CN_SIGMOID; every other combination, and any
 * flag bit an entry point does not define, is rejected (EPS_ERR_INVALID). */
#define EPS_SCORE_KIND_SHIFT 8
#define EPS_SCORE_KIND_MASK (7 << EPS_SCORE_KIND_SHIFT)
#define EPS_SCORE_JACCARD (1 << EPS_SCORE_KIND_SHIFT)
#define EPS_SCORE_SORENSEN (2 << EPS_SCORE_KIND_SHIFT)
#define EPS_SCORE_SALTON (3 << EPS_SCORE_KIND_SHIFT)
#define EPS_SCORE_HUB_PROMOTED (4 << EPS_SCORE_KIND_SHIFT)
#define EPS_SCORE_HUB_DEPRESSED (5 << EPS_SCORE_KIND_SHIFT)
#define EPS_SCORE_LHN (6 << EPS_SCORE_KIND_SHIFT)
#define EPS_SCORE_PREF_ATTACH (7 << EPS_SCORE_KIND_SHIFT)
/* bit k set <=> kind code k (flags >> EPS_SCORE_KIND_SHIFT) is supported; a library without the kinds lacks the
 * symbol, so a stale build fails at load time instead of ignoring the bits */
int eps_score_kinds(void);
int eps_cn_aa(const int32_t *rowptr, const int32_t *col, const float *val, const float *wtable,
              int32_t n, const int32_t *pair_u, const int32_t *pair_v, int64_t M, int flags,
              float *score, int32_t *count, void *workspace, size_t workspace_bytes,
              void *stream);
size_t eps_cn_aa_workspace_bytes(void);

/* ---------------------------------------------------------------------------
 * K2  LinkPredictor MLP over (u,v) Hadamard pairs
 * replaces: LinkGNN.forward's h[edges[0]], h[edges[1]] gathers + LinkPredictor.forward
 *           (/root/reference/models.py:478-485,506).
 *   z0 = h[u] * h[v];  z_{l+1} = relu(W_l z_l + b_l)  (l < L-1);  out = W_{L-1} z + b
 *   score = sigmoid(out) (or the logit when apply_sigmoid == 0)
 * W_h / b_h: HOST arrays of L device pointers; W_l is [out,in] row-major fp32
 * (nn.Linear layout): [H,H] for l < L-1 and [1,H] for the last layer.
 * precision: EPS_MLP_FP32    fp32 FFMA on CUDA cores (reference arithmetic)
 *            EPS_MLP_TC_F16  tcgen05.mma + TMEM: IEEE fp16 operands under a power-of-two scale derived on the
 *                            device from worst-case bounds (no overflow possible; the scale drops out exactly
 *                            at the output layer), fp32 accumulation / output layer / sigmoid.  Needs
 *                            num_layers >= 2, H in {64, 128, 256} and H = 256 -> num_layers <= 3 (the hidden
 *                            layers' weights stay resident in shared memory); EPS_ERR_UNSUPPORTED otherwise
 *                            (e.g. H = 300 of the email config: use EPS_MLP_FP32).
 * ------------------------------------------------------------------------- */
#define EPS_MLP_FP32 0
#define EPS_MLP_TC_F16 1
#define EPS_MLP_TC_BF16 EPS_MLP_TC_F16 /* round-1 name of the tensor-core arm (its operands were bf16 then) */
/* OR-ed into `precision` with EPS_MLP_TC_F16: `workspace` is the buffer of an EARLIER call with the same h
 * (contents), weights, n, H and L, and both calls have M >= 2n (the fp16 copy of h exists) — the scale, the fp16 table
 * and the weight images in it are reused instead of rebuilt (one filter job scores ~100 slabs against the
 * same embeddings).  For M >= 2n, eps_linkpred_workspace_bytes(n, H, L, M, EPS_MLP_TC_F16) and the workspace
 * layout depend on (n, H, L) only, so one buffer sized by any call of the series serves all of them. */
#define EPS_MLP_REUSE_WORKSPACE 0x100
int eps_linkpred_mlp(const float *h, int32_t n, int32_t H, const int32_t *pair_u,
                     const int32_t *pair_v, int64_t M, const float *const *W_h,
                     const float *const *b_h, int32_t L, int precision, int apply_sigmoid,
                     float *score, void *workspace, size_t workspace_bytes, void *stream);
size_t eps_linkpred_workspace_bytes(int32_t n, int32_t H, int32_t L, int64_t M, int precision);

/* ---------------------------------------------------------------------------
 * K7  pair Hadamard gather (training mode of the LinkPredictor) and its backward
 * replaces: h[edges[0]], h[edges[1]] (/root/reference/models.py:506) and x_i * x_j
 *           (/root/reference/models.py:479) inside the training forward
 *           (/root/reference/train_and_eval.py:60-66), and their autograd backward.
 *   forward : out[b,:] = h[pair_u[b],:] * h[pair_v[b],:]              out fp32 [M,H]
 *   backward: dh[pair_u[b],:] += dz[b,:] * h[pair_v[b],:]
 *             dh[pair_v[b],:] += dz[b,:] * h[pair_u[b],:]              dh fp32 [n,H], caller-zeroed, fp32 atomics
 * H must be a multiple of 4.
 * ------------------------------------------------------------------------- */
int eps_pair_hadamard_f32(const float *h, int32_t n, int32_t H, const int32_t *pair_u, const int32_t *pair_v,
                          int64_t M, float *out, void *stream);
int eps_pair_hadamard_bwd_f32(const float *h, int32_t n, int32_t H, const int32_t *pair_u, const int32_t *pair_v,
                              int64_t M, const float *dz, float *dh, void *stream);

/* ---------------------------------------------------------------------------
 * K4  top-k proposal selection
 * replaces: all_scores[:,2].sort(descending=True) + row gather
 *           (/root/reference/filter.py:160-161) followed by the prefix read
 *           (/root/reference/rank.py:294).
 * Radix-select of the k-th score, ordered compaction, stable LSD sort of the
 * k survivors.  Order contract: score descending, ties by position ascending
 * (== torch.sort(descending=True, stable=True)); -0.0 == +0.0; NaN first.
 *   out_idx[j]   = position in `score` of the j-th best element (uint32)
 *   out_score[j] = score[out_idx[j]]
 * Requires 1 <= k <= M < 2^32 - 1.
 * ------------------------------------------------------------------------- */
int eps_topk_f32(const float *score, int64_t M, int64_t k, uint32_t *out_idx, float *out_score,
                 void *workspace, size_t workspace_bytes, void *stream);
size_t eps_topk_workspace_bytes(int64_t M, int64_t k);

/* ---------------------------------------------------------------------------
 * helpers used by the filter driver (filter.py:113-121 packing)
 *   eps_pack_edges: out[j] = (float)u[idx[j]], (float)v[idx[j]], score[j]  -> [k,3] fp32
 * ------------------------------------------------------------------------- */
int eps_pack_edges(const int32_t *pair_u, const int32_t *pair_v, const uint32_t *idx,
                   const float *score, int64_t k, float *out_k3, void *stream);

/* ---------------------------------------------------------------------------
 * K4 over owner slabs: the running proposal set.
 * replaces: the same global sort (filter.py:160-161) when the candidates are
 *           produced slab by slab and never materialised together.
 *   eps_topk_select2_f32: selection (K4 steps 1-3, no sort) over the virtual
 *     concatenation score_a[Ma] ++ score_b[Mb] — a = the running list in
 *     position order, b = the new slab.  out_idx[k] = the positions of the k
 *     best (ties by position) in ASCENDING POSITION order, out_score[k] their
 *     scores.  Position order is all the next call needs, so the running list
 *     is sorted only once, at the end (eps_topk_f32 with k == M).
 *     kth_key_out (device uint32, optional) receives the order key of the k-th
 *     selected score; passed back as prune_key to the NEXT call (valid only when
 *     score_a is that call's full k-element result) it lets the first histogram
 *     pass skip every element that is already worse than the running k-th.
 *   eps_gather_pairs2: (u, v) of those positions from the two pair segments.
 * Workspace: eps_topk_workspace_bytes(Ma + Mb, k).
 * ------------------------------------------------------------------------- */
int eps_topk_select2_f32(const float *score_a, int64_t Ma, const float *score_b, int64_t Mb, int64_t k,
                         const uint32_t *prune_key, uint32_t *kth_key_out, uint32_t *out_idx,
                         float *out_score, void *workspace, size_t workspace_bytes, void *stream);
int eps_gather_pairs2(const int32_t *ua, const int32_t *va, int64_t Ma, const int32_t *ub,
                      const int32_t *vb, const uint32_t *idx, int64_t k, int32_t *out_u, int32_t *out_v,
                      void *stream);

/* ---------------------------------------------------------------------------
 * K4b  threshold push-down: ordered compaction of a slab under the running k-th score
 * replaces: the same global sort (filter.py:160-161).  Once the running list
 *           holds k candidates, only slab elements that beat its k-th score
 *           can enter it; selecting them with one counting read and one
 *           writing read replaces the five radix-select reads of the slab.
 *   bound_key  device uint32: order key of the k-th score s_k (kth_key_out of
 *              eps_topk_select2_f32)
 *   inclusive == 0 : survive iff score > s_k STRICTLY — a slab tie at s_k comes
 *                    later in candidate order than every tie already in the
 *                    list, so by the tie rule it can never displace one
 *   inclusive != 0 : survive iff score >= s_k - margin (margin >= 0): the
 *                    prefilter band of the bf16 tensor-core arm, whose
 *                    survivors are re-scored in fp32 (filter_step.py)
 *   count: tile_offsets[eps_threshold_tiles(M) + 1] (device) = exclusive scan of
 *          the per-tile survivor counts; the last entry is the total, which the
 *          host reads to size the outputs
 *   write: the survivors in POSITION ORDER: (u, v), score and/or position
 *          (any of out_u+out_v / out_score / out_pos may be NULL)
 * eps_topk_select2_f32 with out_idx == out_score == NULL and kth_key_out set
 * returns only the k-th key (re-thresholding of a band pool).
 * ------------------------------------------------------------------------- */
int64_t eps_threshold_tiles(int64_t M);
size_t eps_threshold_workspace_bytes(int64_t M);
int eps_threshold_count(const float *score, int64_t M, const uint32_t *bound_key, float margin,
                        int inclusive, uint32_t *tile_offsets, void *workspace, size_t workspace_bytes,
                        void *stream);
int eps_threshold_write(const float *score, const int32_t *pair_u, const int32_t *pair_v, int64_t M,
                        const uint32_t *bound_key, float margin, int inclusive,
                        const uint32_t *tile_offsets, int32_t *out_u, int32_t *out_v, float *out_score,
                        uint32_t *out_pos, void *stream);

/* ---------------------------------------------------------------------------
 * K4c  segmented top-m select: per-owner proposal budgets
 * replaces: no reference counterpart (the reference keeps a global sort,
 *           filter.py:160-161); "the m best new edges of every node" from one
 *           pass over each owner slab instead of a sort of all candidates.
 * Segments are given by seg_offsets int64[n_seg + 1] (device): segment s is
 * score[seg_offsets[s] .. seg_offsets[s+1]), nondecreasing, seg_offsets[0] == 0
 * and seg_offsets[n_seg] == M (an owner slab's offsets_out of
 * eps_twohop_onepass).  Keys and tie rule are K4's: score descending, ties by
 * position ascending, -0.0 == +0.0.
 *   band == 0 (exact): keep the m best elements of every segment (all of a
 *              segment of <= m elements) - every element whose key is below the
 *              segment's m-th key, plus the first r elements tied with it.
 *   band != 0 : keep every element with score >= s_m - margin (margin >= 0,
 *              s_m = the segment's m-th best score), bounded exactly as K4b's
 *              inclusive threshold (one ulp of slack below the rounded
 *              difference); a segment of <= m elements is kept whole.
 *   select: out_offsets uint32[n_seg + 1] (caller-owned, device) = exclusive
 *           scan of the per-segment kept counts; out_offsets[n_seg] is the
 *           survivor count S, which the host reads to size the outputs.
 *   write : the survivors (u, v, score) in POSITION ORDER, segment s at
 *           out_offsets[s]; out_u / out_v / out_score hold S elements.
 * The per-segment results of select live in the workspace
 * (eps_segment_topk_workspace_bytes(n_seg) bytes, caller-owned) and are read
 * by write: pass the same, unmodified workspace to both calls, in stream order.
 * Requires M < 2^32 - 1, 1 <= m < 2^32 - 1.
 * ------------------------------------------------------------------------- */
size_t eps_segment_topk_workspace_bytes(int64_t n_seg);
int eps_segment_topk_select(const float *score, int64_t M, const int64_t *seg_offsets, int64_t n_seg,
                            int64_t m, float margin, int band, uint32_t *out_offsets, void *workspace,
                            size_t workspace_bytes, void *stream);
int eps_segment_topk_write(const float *score, const int32_t *pair_u, const int32_t *pair_v, int64_t M,
                           const int64_t *seg_offsets, int64_t n_seg, const uint32_t *out_offsets,
                           int32_t *out_u, int32_t *out_v, float *out_score, void *workspace,
                           size_t workspace_bytes, void *stream);

/* ---------------------------------------------------------------------------
 * K6 / K6+K3  2-hop candidates of the owner range [v_lo, v_hi), optionally
 * TOGETHER WITH their CN / AA / RA scores from one walk over the 2-paths of
 * each owner, without a count pass.
 * replaces: A2 = adj_t @ adj_t; remove_diag; A2[adj>0] = 0; nonzero
 *           (/root/reference/filter.py:96-109, CPU, single thread; the A@A
 *           values are discarded at :108-109) + the scoring loop
 *           filter.py:113-142 for the heuristic models (models.py:536-554,
 *           adamic_utils.py:13-25, train_and_eval.py:195-216).
 * Candidates of owner v (= all_edges[:,1]) are every u != v with a common
 * neighbour and no edge (u,v); they are emitted in ascending u, owners in
 * ascending v: the reference's column-major order, no sort needed.
 * A2's values ARE the scores: each 2-path v-k-u adds 1 (CN) or wtable[k]
 * (AA: 1/log deg, RA: 1/deg) to candidate (u, v).  Sums are accumulated as
 * 64-bit fixed-point integers with atomics (exact, order-independent), so
 * score[i] == eps_cn_aa's score of the same pair, bit for bit.
 * Every owner writes into a padded slot sized by a cheap upper bound of its
 * candidate count and records its real count; a scan of the counts and a
 * compaction pass (fixed point -> fp32, which reads every accumulator anyway)
 * move the results to their compact positions.  No inter-CTA dependency.
 *   bound_offsets int64[v_hi - v_lo + 1] (device): exclusive prefix of any
 *                upper bound of the per-owner candidate counts, e.g.
 *                min(#2-paths(v), n - 1 - deg(v)); bound_offsets[last] == cap.
 *                An owner whose real count exceeded its bound would write
 *                into its neighbour's slot: the bound must hold.
 *   cap          capacity (in candidates) of pair_u / pair_v / score / count
 *   offsets_out  int64[v_hi - v_lo + 1] (device): exclusive prefix of the
 *                real per-owner counts; offsets_out[last] = N <= cap, and the
 *                first N entries of the outputs are valid.
 *   val          fp32[nnz] edge values or NULL (all ones).  With values (collab)
 *                a 2-path v-k-u contributes A[u,k] * (A[v,k] * wtable[k]) (or
 *                A[u,k] * A[v,k] without wtable) — eps_cn_aa's products; the
 *                kernel reads A[k,u] for A[u,k], so A must be bitwise symmetric.
 *   wtable       NULL -> score = CN count; else score = sum of wtable[k]
 *   flags        EPS_CN_SIGMOID | a similarity kind (EPS_SCORE_*, see eps_cn_aa;
 *                degrees from rowptr) | EPS_TWOHOP_UPPER
 *   score        fp32[cap] or NULL;  count int32[cap] or NULL (exact CN).
 *                score == NULL and count == NULL -> enumeration only (the GNN
 *                filter models).  A similarity kind runs the count-only walk
 *                and applies its formula in the compaction pass: weighted
 *                graphs pass val == NULL (structure only).
 *   flags |= EPS_TWOHOP_UPPER: upper-triangle mode, only the candidates u > v
 *                of every owner v (each unordered pair once, under its smaller
 *                end).  Both walks visit only the suffix u > v of every N(k)
 *                and the bitmap work starts at word (v + 1) / 32; the bound
 *                may then be min(#2-paths v-k-u with u > v,
 *                n - 1 - v - |N(v) & (v, n)|).  Owner v's output is (u, v) in
 *                ascending u, and every score equals the full kernel's score
 *                of the same pair, bit for bit.
 * Needs ~3n/16 bytes of shared memory (<= 200 KB, i.e. n <= ~1.0M).
 * ------------------------------------------------------------------------- */
#define EPS_TWOHOP_UPPER 4
int eps_twohop_onepass(const int32_t *rowptr, const int32_t *col, const float *val, const float *wtable,
                       int32_t n, int32_t v_lo, int32_t v_hi, const int64_t *bound_offsets, int64_t cap, int flags,
                       int32_t *pair_u, int32_t *pair_v, float *score, int32_t *count,
                       int64_t *offsets_out, void *workspace, size_t workspace_bytes, void *stream);
size_t eps_twohop_onepass_workspace_bytes(int64_t cap, int32_t n_owners);

/* ---------------------------------------------------------------------------
 * Local Path index  LP(u, v) = (A^2)_uv + 1e-3 * (A^3)_uv   (Lue & Zhou)
 * replaces: no reference counterpart (a heuristic filter / rank model of this
 *           project, 'local_path').  Structure only: N(x) is the stored list
 *           (self loops included), edge values are ignored.
 *   c2 = |N(u) & N(v)|,  c3 = sum_{j in N(u)} |N(j) & N(v)|   (exact int32: c3 <= nnz < 2^31)
 *   score = __double2float_rn(__dadd_rn((double)c2, __dmul_rn(1e-3, (double)c3)))
 * The adjacency must be structurally symmetric ((u,k) stored <=> (k,u) stored,
 * no repeated entry); the caller checks it.
 *
 * eps_local_path_onepass: the eps_twohop_onepass contract (padded slots sized
 *   by bound_offsets / cap, per-owner counts, offsets_out, heaviest owners
 *   first, EPS_TWOHOP_UPPER) for the Local Path score, from one fused walk.
 *   tri        int32[nnz]: tri[p] = |N(v) & N(col[p])| for the stored arc p of
 *              row v (eps_cn_aa counts of the pairs (col[p], v))
 *   max_count  an upper bound of EVERY owner's full candidate count (u > v
 *              or not) in [v_lo, v_hi); sizes the per-CTA c2 scratch
 *   ctas       number of per-CTA scratch areas in the workspace; the kernel
 *              runs at most that many CTAs
 *   flags      0 or EPS_TWOHOP_UPPER (only u > v is emitted; bound_offsets
 *              then bound the half counts)
 *   score / c2 / c3  fp32 / int32 / int32 [cap] or NULL each
 * Workspace: eps_local_path_onepass_workspace_bytes(cap, v_hi - v_lo, max_count, ctas).
 *
 * eps_local_path_pairs: c2, c3 and the score of any pair list (u == v, edges
 *   and isolated ends included).  One CTA holds the N(v) bitmap per run of
 *   equal pair_v; a pair costs sum_{j in N(u)} deg j, so sort the pairs by v
 *   and keep this for evaluation sets.  flags must be 0.
 * Both need n/8 + ... bytes of shared memory (<= 200 KB) like the K6 kernels.
 * ------------------------------------------------------------------------- */
int eps_local_path_onepass(const int32_t *rowptr, const int32_t *col, const int32_t *tri, int32_t n, int32_t v_lo,
                           int32_t v_hi, const int64_t *bound_offsets, int64_t cap, int64_t max_count, int32_t ctas,
                           int flags, int32_t *pair_u, int32_t *pair_v, float *score, int32_t *c2, int32_t *c3,
                           int64_t *offsets_out, void *workspace, size_t workspace_bytes, void *stream);
size_t eps_local_path_onepass_workspace_bytes(int64_t cap, int32_t n_owners, int64_t max_count, int32_t ctas);
int eps_local_path_pairs(const int32_t *rowptr, const int32_t *col, int32_t n, const int32_t *pair_u,
                         const int32_t *pair_v, int64_t M, int flags, float *score, int32_t *c2, int32_t *c3,
                         void *workspace, size_t workspace_bytes, void *stream);
size_t eps_local_path_pairs_workspace_bytes(void);

/* ---------------------------------------------------------------------------
 * K6 at distance 3: the distance-<= 3 candidates of the owner range [v_lo, v_hi)
 * replaces: no reference counterpart (the reference enumerates 2-hop pairs
 *           only, filter.py:96-109); proposal sets for the GNN filters that
 *           include pairs without a common neighbour.
 * Candidates of owner v are every u with (A^2)_uv + (A^3)_uv > 0 that is
 * neither v nor in N(v): the ends of 2-walks and 3-walks from v (stored lists,
 * self loops included, edge values ignored).  The 2-hop set of
 * eps_twohop_onepass is a subset.  Enumeration only; owners ascending,
 * candidates ascending in u (column-major order).
 * The eps_twohop_onepass contract: padded slots sized by bound_offsets / cap
 * (any upper bound of the per-owner counts, e.g. min(#2-walks + #3-walks,
 * n - 1 - deg v + [self loop])), offsets_out, heaviest owners first,
 * EPS_TWOHOP_UPPER (only u > v; the bounds then bound the half counts), and a
 * violated bound poisons N (offsets_out[last] > cap) instead of overrunning.
 *   max_ends   an upper bound of EVERY owner's number of distinct 2-walk ends
 *              in [v_lo, v_hi) (e.g. min(#2-walks, n)); sizes the per-CTA list
 *              the kernel freezes them in
 *   ctas       number of per-CTA lists in the workspace; the kernel runs at
 *              most that many CTAs
 *   flags      0 or EPS_TWOHOP_UPPER
 * Every argument is checked before any CUDA call.
 * Workspace: eps_threehop_onepass_workspace_bytes(cap, v_hi - v_lo, max_ends, ctas).
 * Needs ~3n/16 bytes of shared memory (<= 200 KB, i.e. n <= ~1.0M), as K6.
 * ------------------------------------------------------------------------- */
int eps_threehop_onepass(const int32_t *rowptr, const int32_t *col, int32_t n, int32_t v_lo, int32_t v_hi,
                         const int64_t *bound_offsets, int64_t cap, int64_t max_ends, int32_t ctas, int flags,
                         int32_t *pair_u, int32_t *pair_v, int64_t *offsets_out, void *workspace,
                         size_t workspace_bytes, void *stream);
size_t eps_threehop_onepass_workspace_bytes(int64_t cap, int32_t n_owners, int64_t max_ends, int32_t ctas);

/* ---------------------------------------------------------------------------
 * K5  multi-GPU merge of per-GPU proposal lists (no counterpart in the
 * single-GPU reference; SURVEY.md section 8e).  One ncclAllGather of the
 * [k_local,3] fp32 (u, v, score) rows of every rank followed by a K4 select
 * over the world*k_local gathered rows, executed identically on every rank.
 * Ranks must own ascending, contiguous owner ranges so that position in the
 * gathered array preserves the global tie order.  Pad short local lists with
 * score = -inf rows.  eps_comm_* wrap ncclGetUniqueId / ncclCommInitRank
 * (resolved by dlopen of libnccl.so.2); id buffers are 128-byte HOST buffers.
 * ------------------------------------------------------------------------- */
int eps_comm_unique_id(void *out128_h);
int eps_comm_init(const void *id128_h, int world, int rank, void **comm_out);
int eps_comm_destroy(void *comm);
int eps_topk_merge_allgather(void *comm, const float *local_k3, int64_t k_local, int64_t k,
                             float *out_k3, void *workspace, size_t workspace_bytes, void *stream);
size_t eps_topk_merge_workspace_bytes(int world, int64_t k_local, int64_t k);

#ifdef __cplusplus
}
#endif
#endif /* EPS_B200_H */
