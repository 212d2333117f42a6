/*
 * rtucker.h -- C ABI of librtucker_b200.so: the B200 (sm_100a) hot path of R-TuckER.
 *
 * The reference (johanDDC/R-TuckER) is pure Python and has no FFI layer; each entry point
 * below names the reference file:line whose arithmetic it replaces.  A maintainer binds
 * them with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; rt_last_error() returns a
 *     thread-local, NUL-terminated description of the last failure on the calling thread;
 *   - no C++ types, exceptions or torch types cross this boundary;
 *   - every pointer is a DEVICE pointer owned by the caller unless the name ends in _host;
 *     inputs, outputs and workspaces are all caller-allocated (query *_ws_bytes first);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*): no hidden
 *     synchronisation, no hidden allocation, nothing retained after return;
 *   - matrices are row-major fp32 with an explicit leading dimension (in elements) where
 *     one is given, otherwise dense; indices are int32; "small" matrices produced by the
 *     N-independent stage are fp64;
 *   - hyper-parameters that change between steps live in device memory (`hyper`), so a
 *     captured CUDA graph of a step stays valid:  hyper[0]=lr, hyper[1]=reg,
 *     hyper[2]=momentum_beta, hyper[3]=normalize_grad (0 => do not normalise).
 *   - mode order is (relation, subject, object) as in train.py:37-42; ranks (r0,r1,r2);
 *     `sym` != 0 selects the SF-Tucker manifold (subject and object share the factor E,
 *     r1 == r2).
 */
#ifndef RTUCKER_H_
#define RTUCKER_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_ABI_VERSION 1

/* ---- library ------------------------------------------------------------------------- */
int rt_abi_version(void);
const char* rt_last_error(void);
/* SM count and compute capability of the current device. */
int rt_device_info(int* sm_count_host, int* cc_major_host, int* cc_minor_host);
/* Number of CUDA kernels this library has launched in the calling process (bench.py: gpu_launches). */
unsigned long long rt_launch_count(void);

/* ---- (d) filtered ranking ------------------------------------------------------------ */
/*
 * Replaces filter_predictions (src/utils/utils.py:15-22) + metrics (src/utils/metrics.py:4-8)
 * on a dense prediction matrix P[B, ldp>=N] (the reference's own probabilities).
 * For query b with target column t=target[b] and filter list F_b = flt_idx[flt_off[b]:flt_off[b+1]]
 * (all known true objects of (s,r); may or may not contain t):
 *     p'_j = 0 for j in F_b \ {t},   p'_j = P[b,j] otherwise
 *     greater[b]      = #{ j != t : p'_j >  P[b,t] }
 *     equal[b]        = #{ j != t : p'_j == P[b,t] }
 *     equal_before[b] = #{ j <  t : p'_j == P[b,t] }
 * The reference's rank is 1 + greater + (position of t among its ties, implementation defined
 * by torch.sort); 1 + greater + equal_before is the stable-sort rank.
 */
int rt_rank_filtered(const float* P, int64_t ldp, int B, int N,
                     const int32_t* target, const int32_t* flt_off, const int32_t* flt_idx,
                     int32_t* greater, int32_t* equal, int32_t* equal_before, void* stream);

/*
 * Same counts without materialising P:  P[b,j] = sigmoid(q[b,:] . O[j,:]) in fp32
 * (src/model/asymmetric/R_TuckER.py:47-48 fused with the ranking above).  O is an entity
 * shard holding global rows [n_begin, n_begin+n_local); p_target[b] is the target's
 * probability (computed by the shard that owns it with rt_target_prob and shared by the
 * caller).  Counts are shard-local partial sums (sum them over shards).
 * bce_sum (double[1], may be NULL) accumulates the un-smoothed BCE of train.py:113 over the
 * shard: sum_{b,j} -(t log p + (1-t) log(1-p)) with t = 1 on the filter list.
 */
int rt_target_prob(const float* q, const float* O, int B, int r2, int n_begin, int n_local,
                   const int32_t* target, float* p_target, void* stream);
size_t rt_score_rank_ws_bytes(int B, int n_local, int r2);
int rt_score_rank_fused(const float* q, const float* O, int B, int r2, int n_begin, int n_local,
                        const int32_t* target, const float* p_target,
                        const int32_t* flt_off, const int32_t* flt_idx,
                        int32_t* greater, int32_t* equal, int32_t* equal_before,
                        double* bce_sum, void* ws, void* stream);

/*
 * Filtered top-k link prediction without materialising P: which k entities best complete (s, r, ?).
 * q[B, r2] are the query rows (rt_query_fwd), O the entity shard holding global rows [n_begin, n_begin+n_local).
 * For query b, with filter list F_b = flt_idx[flt_off[b]:flt_off[b+1]] (global ids, ASCENDING within each query, as
 * the data pipeline produces them; flt_off and flt_idx both NULL: no filtering):
 *     p_j = sigmoid(q_b . O_j), bit-identical to rt_score_dense;  entities in F_b are excluded;
 *     order: p descending, then global id ascending (a total order: the entity at position i has filtered rank i + 1
 *            under rt_rank_filtered / rt_score_rank_fused whenever its p > 0);
 *     top_idx[b, 0:k] (int32 global ids), top_p[b, 0:k] (the exact p).  Positions beyond the number of unfiltered
 *            entities of the shard get id -1 and p = -inf, so per-shard lists merge without special cases.
 * n_cand[b] (may be NULL) tells which path produced query b: >= 0 the number of tensor-core candidates that were
 * rechecked exactly, -1 the exact full pass.  The path is chosen from the shape and from device flags only.
 * Limits: 1 <= k <= 256, 1 <= B <= 1024 per call, 1 <= r2 <= 256; anything else returns an error.
 * The workspace (rt_score_topk_ws_bytes) does not grow with n_local beyond the shard's row norms and a fixed chunk:
 * tens of MB at B = 512, n_local = 10^6, r2 = 200, k = 100 instead of the 2 GB of the dense probabilities.
 */
size_t rt_score_topk_ws_bytes(int B, int n_local, int r2, int k);
int rt_score_topk(const float* q, const float* O, int B, int r2, int n_begin, int n_local, int k,
                  const int32_t* flt_off, const int32_t* flt_idx,
                  int32_t* top_idx, float* top_p, int32_t* n_cand, void* ws, void* stream);

/* Dense compatibility path: P[b, j] = sigmoid(q_b . O_j), what score_fn(T) returns in the reference
 * (src/model/asymmetric/R_TuckER.py:47-48).  Bit-identical to the values the fused kernels use. */
int rt_score_dense(const float* q, const float* O, int B, int r2, int n_local, float* P, int64_t ldp,
                   void* stream);
/* In-place dense filter, exactly src/utils/utils.py:18-21 (filter_col = features[:,2]). */
int rt_filter_dense(float* P, int64_t ldp, float* T, int64_t ldt, int B, int N,
                    const int32_t* filter_col, void* stream);

/* ---- (d') evaluation and prediction in logit space ----------------------------------- */
/*
 * For models trained with the softmax cross-entropy (rt_score_ce_fwd_bwd), whose top logits sit where the fp32 sigmoid
 * has saturated (p == 1.0f from z = 16.6 on, coarse steps of p well below): ranks and top-k on the exact fp32 logit
 * z_bj = q_b . O_j (k ascending, one fmaf accumulator: the value rt_score_dense passes to the sigmoid) instead of p.
 *
 * rt_score_dense_logits: Z[b, j] = z_bj, bit-identical to the logits inside rt_score_dense.
 * rt_target_logit: z_target[b] = z_{b, target[b]} on the shard that owns the target, 0 elsewhere (sum over shards).
 * rt_score_rank_logit: filtered counts in logit space, as shard partial sums.  Filtered entities are REMOVED (not
 *   scored 0 as in rt_score_rank_fused: 0 is an ordinary logit).  With F_b = flt_idx[flt_off[b]:flt_off[b+1]] (global
 *   ids, unique; flt_off and flt_idx both NULL: no filter), t = target[b], zt = z_target[b] (summed over shards):
 *     greater[b]      = #{ j in shard, j not in F_b, j != t : z_bj >  zt }
 *     equal[b]        = #{ j in shard, j not in F_b, j != t : z_bj == zt }
 *     equal_before[b] = the same as equal, restricted to j < t           (rank = 1 + greater + equal_before)
 *     pos_sum[b]      = sum_{j in F_b and in shard} z_bj (double; pos_sum may be NULL), summed in a fixed order.
 *   With lse_b from rt_score_lse, lse_b - pos_sum[b] / |F_b| is the cross-entropy of the un-smoothed multi-hot target
 *   y / |y|.  Limits: 1 <= B <= 65535, 1 <= r2 <= 256.  Deterministic; no host synchronisation.
 * rt_score_topk_logit: rt_score_topk (same arguments, limits and workspace, rt_score_topk_ws_bytes) with z in place of
 *   p: order z descending, then global id ascending; top_z the exact z, bit-identical to rt_score_dense_logits;
 *   padding id -1, z = -inf.
 */
int rt_score_dense_logits(const float* q, const float* O, int B, int r2, int n_local, float* Z, int64_t ldz,
                          void* stream);
int rt_target_logit(const float* q, const float* O, int B, int r2, int n_begin, int n_local,
                    const int32_t* target, float* z_target, void* stream);
size_t rt_score_rank_logit_ws_bytes(int B, int n_local, int r2);
int rt_score_rank_logit(const float* q, const float* O, int B, int r2, int n_begin, int n_local,
                        const int32_t* target, const float* z_target,
                        const int32_t* flt_off, const int32_t* flt_idx,
                        int32_t* greater, int32_t* equal, int32_t* equal_before,
                        double* pos_sum, void* ws, void* stream);
int rt_score_topk_logit(const float* q, const float* O, int B, int r2, int n_begin, int n_local, int k,
                        const int32_t* flt_off, const int32_t* flt_idx,
                        int32_t* top_idx, float* top_z, int32_t* n_cand, void* ws, void* stream);

/* ---- (a) query contraction ----------------------------------------------------------- */
/* out[b,:] = table[idx[b] - row_begin, :] if row_begin <= idx[b] < row_begin+rows else 0.
 * Replaces the gathers at src/model/asymmetric/R_TuckER.py:43-44 (shard-aware). */
int rt_gather_rows(const float* table, int rows, int r, int row_begin,
                   const int32_t* idx, int B, float* out, void* stream);
/* rows of `rows_in[B,r]` are added into table[idx[b]-row_begin] (owner shard only), duplicates
 * summed in ascending b (deterministic).  Used for the sparse part of dV_S / dV_R. */
int rt_scatter_rows_add(float* table, int rows, int r, int row_begin,
                        const int32_t* idx, int B, const float* rows_in, void* stream);

/* q[b,:] = core x_1 r_rows[b] x_2 s_rows[b]        (R_TuckER.py:45-46: einsum + bmm). */
size_t rt_query_ws_bytes(int B, int r0, int r1, int r2);
int rt_query_fwd(const float* core, const float* r_rows, const float* s_rows,
                 int B, int r0, int r1, int r2, float* q, void* ws, void* stream);
/* Backward of the above given H = dL/dq [B,r2] (what autograd does for R_TuckER.py:45-46):
 * d_core[r0,r1,r2] = sum_b r_b (x) s_b (x) H_b;  ds_rows[B,r1];  dr_rows[B,r0]. */
int rt_query_bwd(const float* core, const float* r_rows, const float* s_rows, const float* H,
                 int B, int r0, int r1, int r2,
                 float* d_core, float* ds_rows, float* dr_rows, void* ws, void* stream);
/* t[b,:] = core x_2 s_rows[b] x_3 o_rows[b]: t[b,a] = sum_{i,j} core[a,i,j] s_rows[b,i] o_rows[b,j]  [B, r0].
 * The relation-mode query of relation prediction (s, ?, o): z_bm = R[m] . t_b scores every relation, so the
 * entity-side ranking, top-k and log-sum-exp entry points take t as the query rows and the relation factor as O.
 * Reads the core in place (no permuted copy).  Bit-identical to rt_query_fwd on core permuted to (r1, r2, r0)
 * with (s_rows, o_rows) in place of (r_rows, s_rows): same products, same split plan, same summation order.
 * Deterministic; B == 0 launches nothing. */
size_t rt_pair_ws_bytes(int B, int r0, int r1, int r2);
int rt_pair_fwd(const float* core, const float* s_rows, const float* o_rows,
                int B, int r0, int r1, int r2, float* t, void* ws, void* stream);
/* Backward of rt_pair_fwd given H_t = dL/dt [B, r0] (the relation-prediction term of the training step):
 * d_core[r0,r1,r2] = sum_b H_t[b] (x) s_rows[b] (x) o_rows[b];
 * ds_rows[b,i] = sum_{a,j} core[a,i,j] H_t[b,a] o_rows[b,j]  [B, r1];
 * do_rows[b,j] = sum_{a,i} core[a,i,j] H_t[b,a] s_rows[b,i]  [B, r2].
 * Reads the core in place and writes d_core unpermuted (no permuted copies).  Bit-identical to rt_query_bwd on core
 * permuted to (r1, r2, r0) with (s_rows, o_rows, H_t) in place of (r_rows, s_rows, H), its d_core permuted back, its
 * ds_rows as do_rows and its dr_rows as ds_rows: same products, same split plan, same summation order.
 * The workspace of rt_pair_ws_bytes covers both passes.  Deterministic; B == 0 launches nothing. */
int rt_pair_bwd(const float* core, const float* s_rows, const float* o_rows, const float* H_t,
                int B, int r0, int r1, int r2,
                float* d_core, float* ds_rows, float* do_rows, void* ws, void* stream);

/* ---- (b) fused 1-N score + sigmoid + label-smoothed BCE + backward ------------------- */
/*
 * Replaces R_TuckER.py:47-48 (q @ O^T, sigmoid), nn.BCELoss(mean) at train.py:79,136 with the
 * dense label-smoothed targets of src/data/Dataset.py:43-52, and their autograd backward.
 * The B x N logit / probability / target matrices are never written to memory.
 *   Z = q O^T,  P = sigmoid(Z),  T[b,j] = (1-ls)*[j in tgt(b)] + ls/n_total
 *   loss_sum = sum_{b,j} -(T max(log P,-100) + (1-T) max(log1p(-P),-100))
 *   G = (P-T)/max(P(1-P),1e-12) * P(1-P) * 1/(B_total*n_total)
 *   H  = G O        [B, r2]   (shard partial)
 *   dO = G^T qp     [n_local, r2]      (qp = q for the raw partial; pass q.A to fold a right factor)
 * O holds global entity rows [n_begin, n_begin+n_local); tgt_idx holds GLOBAL entity ids.
 * loss_sum is a double[1] (un-normalised sum over the shard; divide by B_total*n_total).
 * variant: 0 = fp32 FFMA (parity path),
 *          2 = warp-specialised tcgen05 kernel with power-of-two-scaled fp16 operands (same 11 significant
 *              bits as TF32, stated tolerance 2e-3); qp must be NULL or q (dO = G^T q).
 *          Any other variant returns an error (the 3xTF32 tensor-core path is rt_score_bce_tc3).
 */
size_t rt_score_bce_ws_bytes(int B, int n_local, int r2, int variant);
int rt_score_bce_fwd_bwd(const float* q, const float* qp, const float* O,
                         int B, int r2, int n_begin, int n_local, int n_total, int b_total,
                         const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing,
                         double* loss_sum, float* H, float* dO,
                         int variant, void* ws, void* stream);
/* Variant 2 called directly.  o_absmax_hint > 0 promises max |O| <= hint (1.0 for the orthonormal factors of a
 * point on the manifold) and saves the pass that measures it; <= 0 measures it on the device.
 * centre_state (device float[2], may be NULL): [1] = the mean of p - t measured by the previous call (caller-owned,
 * persistent across steps; initialise to 0.5).  The fp16 gradient operand G is stored centred by that value and the
 * rank-one part is added back exactly in fp32: without it the 11-bit operand rounds away the 1e-4 deviations of
 * p around 0.5 that carry the whole signal at the start of training (measured: no learning from the xavier/QR
 * initialisation).  NULL = no centring. */
int rt_score_bce_v3_supported(int r2);
size_t rt_score_bce_v3_ws_bytes(int B, int n_local, int r2);
int rt_score_bce_v3(const float* q, const float* O, int B, int r2, int n_begin, int n_local, int n_total,
                    int b_total, const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing,
                    float o_absmax_hint, double* loss_sum, float* H, float* dO, float* centre_state, void* ws,
                    void* stream);

/* Variant 3: the same operation at fp32 accuracy on the tensor cores (apply_tc.cu, score mode): logits by 3xTF32 with
 * round-to-nearest partial sums, loss and gradient with the fp32 semantics of variant 0, the two backward contractions
 * by the 3xTF32 factor-update kernel.  Like variant 0: dO = G^T qp (qp = q when NULL).  The gradient matrix G (B x n_local fp32) is
 * staged in the workspace between the launches (it fits the 126 MB L2 at WN18RR size); the logit / probability /
 * target matrices never exist. */
int rt_score_bce_tc3_supported(int B, int n_local, int r2);
size_t rt_score_bce_tc3_ws_bytes(int B, int n_local, int r2);
int rt_score_bce_tc3(const float* q, const float* qp, const float* O, int B, int r2, int n_begin, int n_local,
                     int n_total, int b_total, const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing,
                     double* loss_sum, float* H, float* dO, void* ws, void* stream);

/* ---- (b') fused 1-N softmax cross-entropy + backward ------------------------------------ */
/*
 * The other standard objective of 1-N scoring (KvsAll / 1vsAll trainers): softmax cross-entropy over ALL entities.
 * For query b with target set y_b (tgt_idx[tgt_off[b]:tgt_off[b+1]], GLOBAL ids, unique), label smoothing ls,
 * N = n_total entities and logits z_bj = q_b . O_j:
 *   t_bj   = (1 - ls) [j in y_b] / |y_b| + ls / N            (sum_j t_bj = 1)
 *   lse_b  = log sum_j exp(z_bj)                              (over all N entities, all shards)
 *   loss   = (1/B) sum_b (lse_b - sum_j t_bj z_bj) + reg ||core||^2
 *   G_bj   = dloss/dz_bj = (exp(z_bj - lse_b) - t_bj) / B
 * i.e. torch.nn.functional.cross_entropy(z, y / |y|, label_smoothing=ls, reduction="mean").  A query with no targets
 * (|y_b| = 0: the CSR lives on the device and is not checked) is defined, not rejected: its positive term is 0 and
 * only the ls / N part of t remains (loss_b = lse_b - (ls/N) sum_j z_bj, G = (softmax - ls/N) / B).  Correct for
 * any finite fp32 logits (|z| ~ 1e3 included): the max is kept online.
 *
 * Two passes per entity shard (global rows [n_begin, n_begin + n_local)):
 * rt_score_lse: parts[B][2] (fp32) = (m_b, s_b), m_b the largest logit of the shard, s_b = sum_{j in shard}
 *   exp(z_bj - m_b); an empty shard gives (-inf, 0).  No B x N object is written.
 * rt_score_ce_fwd_bwd: parts[nparts][B][2] are the rt_score_lse results of ALL shards (nparts = 1 unsharded), merged
 *   in a fixed order into lse_b.  Outputs as rt_score_bce_fwd_bwd:  H = G O [B, r2] (shard partial),
 *   dO = G^T qp [n_local, r2] (qp = q when NULL), loss_sum (double[1]) = sum_b sum_{j in shard} t_bj (lse_b - z_bj):
 *   un-normalised (divide by b_total); summed over the shards it is B times the loss without the regulariser (the
 *   (1 - ls) lse_b of a query without targets is charged to the shard with n_begin == 0).
 * variant: 0 = fp32 FFMA (any shape), 3 = 3xTF32 tensor cores (the shapes of rt_score_bce_tc3_supported).  Any other
 * variant, or nparts < 1, returns an error.  Deterministic: the same inputs give the same bits.
 */
size_t rt_score_lse_ws_bytes(int B, int n_local, int r2, int variant);
int rt_score_lse(const float* q, const float* O, int B, int r2, int n_local, int variant, float* parts, void* ws,
                 void* stream);
size_t rt_score_ce_ws_bytes(int B, int n_local, int r2, int variant);
int rt_score_ce_fwd_bwd(const float* q, const float* qp, const float* O, int B, int r2, int n_begin, int n_local,
                        int n_total, int b_total, const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing,
                        const float* parts, int nparts, double* loss_sum, float* H, float* dO, int variant, void* ws,
                        void* stream);

/* ---- (c) tall-skinny passes over the N x r factors ----------------------------------- */
/* out[ra, rb] (fp64) = A[n, :ra]^T  B[n, :rb]   (deterministic two-stage reduction).
 * precise = 0: fp32 products accumulated in fp32 over 256-row blocks, fp64 across blocks;
 * precise = 1: exact fp64 accumulation (needed where the Gram feeds a Cholesky: the retraction).
 * Replaces the N-sized Gram products inside tucker_riemopt grad/project/norm/round
 * (call sites asymmetric/optim.py:86-90,108). */
size_t rt_gram_ws_bytes(int n, int ra, int rb);
int rt_gram(const float* A, int64_t lda, const float* B, int64_t ldb, int n, int ra, int rb,
            double* out, int precise, void* ws, void* stream);
/*
 * Y[n, rc] = a0 * X0 + sum_{k<nk} X_k[n, rk_k] . K_k[rk_k, rc]      (K_k fp64, row-major dense)
 * a0 is read from device memory (a0_dev, may be NULL => 1.0 when X0 != NULL).  X0 may be NULL.
 * Y may alias X0 (same ld) but no X_k, k>=1.  Replaces the N-sized factor updates of
 * project / construct / round and the p.data.add_ write-back (asymmetric/optim.py:106-114).
 */
int rt_apply(float* Y, int64_t ldy, int n, int rc,
             const float* X0, int64_t ldx0, const double* a0_dev,
             int nk, const float* const* X_host, const int64_t* ldx_host, const int* rk_host,
             const double* const* K_host, void* stream);

/* Tensor-core (tcgen05, TF32 with a 3-product hi/lo split, partial sums added with round-to-nearest => the accuracy
 * of the FFMA kernel, a few 1e-7) variant of rt_apply.  *_supported returns 1 if the shape fits (width <= 256). */
int rt_apply_tc_supported(int rc, int nk, const int* rk_host);
size_t rt_apply_tc_ws_bytes(int rc, int nk, const int* rk_host);
int rt_apply_tc(float* Y, int64_t ldy, int n, int rc, const float* X0, int64_t ldx0, const double* a0_dev,
                int nk, const float* const* X_host, const int64_t* ldx_host, const int* rk_host,
                const double* const* K_host, void* ws, void* stream);
/* Several independent updates of the same width rc in ONE persistent launch (the subject and the object factor of
 * a step).  Per job: Y = a0 * X0 + sum_t X_t . K_t as above; Y may alias X0 AND any X_t (each row tile is read
 * completely before it is written); copy_out[t] (optional) receives the raw X_t while it streams through -- the
 * "old point" / "kept direction" copies of RSGDwithMomentum.step (asymmetric/optim.py:109-114) without extra passes. */
typedef struct rt_apply_job {
  float* Y; int64_t ldy; int n;
  const float* X0; int64_t ldx0; const double* a0_dev;
  int nk;
  const float* X[4]; int64_t ldx[4]; int rk[4]; const double* K[4];
  float* copy_out[4]; int64_t ldcopy[4];
} rt_apply_job;
size_t rt_apply_multi_ws_bytes(int njobs, const rt_apply_job* jobs, int rc);
int rt_apply_multi(int njobs, const rt_apply_job* jobs, int rc, void* ws, void* stream);

/* ---- (c) N-independent ("small") stage ----------------------------------------------- */
/*
 * All r-sized arithmetic of one optimiser step, in fp64, on a caller-provided workspace.
 * Layout of the workspace is private; sizes come from rt_small_ws_bytes.
 *
 * rt_small_prepare: from core -> Gram of each unfolding S_(i)S_(i)^T (SF: shared modes summed),
 *   their inverses A_i, ||core||^2.        (tucker_riemopt grad's (S_(i)S_(i)^T)^-1 factor)
 *   Ainv2_f32[r2,r2] receives A_2 in fp32 (to fold into qp = q.A_2 with rt_matmul_small).
 */
size_t rt_small_ws_bytes(int r0, int r1, int r2, int B);
int rt_small_prepare(const float* core, int r0, int r1, int r2, int sym,
                     void* small_ws, void* stream);
/* Byte offset inside small_ws of the fp64 matrix A_mode [r_mode, r_mode] written by rt_small_prepare (so the
 * caller can hand it to rt_apply as a right factor). */
size_t rt_small_ainv_offset(int mode, int r0, int r1, int r2);
/* C[m,n] = A[m,k] . (fp64 K from small_ws slot `which`: 0,1,2 = Ainv_0..2), fp32 in/out.  */
int rt_rows_times_ainv(const float* A, int m, int mode, int r0, int r1, int r2,
                       float* C, void* small_ws, void* stream);
/*
 * rt_small_grad: finishes the Riemannian gradient (SURVEY App. A.3) from the kernel outputs.
 *   in : d_core (raw), q, qp(=q.A_2), H, r_rows, s_rows, dr_rows, ds_rows, bce loss_sum,
 *        hyper (reg), b_total*n_total
 *   out: dS_g[r0,r1,r2] fp32 = d_core + 2 reg core;  loss_total (double[1]) = bce + reg||core||^2;
 *        drA[B,r0], dsA[B,r1] fp32 (rows . A_i, to scatter);  fp64 P_i = -(U_i^T g_i A_i):
 *        P_R[r0,r0], P_S[r1,r1], P_O[r2,r2]   (SF: P_S holds the shared one, P_O aliases it)
 */
int rt_small_grad(const float* core, const float* d_core, const float* qp, const float* H,
                  const float* r_rows, const float* s_rows,
                  const float* dr_rows, const float* ds_rows,
                  const double* bce_sum, double inv_count, const double* hyper,
                  int B, int r0, int r1, int r2, int sym,
                  float* dS_g, double* loss_total, float* drA, float* dsA,
                  double* P_R, double* P_S, double* P_O, void* small_ws, void* stream);
/*
 * rt_small_norm: ||xi||^2 = ||dS||^2 + sum_i tr(Gram_i . S_(i)S_(i)^T)  -> norm (double[1]) and
 * alpha (double[1]) = normalize_grad/norm (1 if hyper[3]==0).   (asymmetric/optim.py:90-92)
 * gram_i = dV_i^T dV_i (fp64, from rt_gram; SF: gram_S is the shared one, gram_O ignored).
 */
int rt_small_norm(const float* dS_g, const double* gram_R, const double* gram_S, const double* gram_O,
                  const double* hyper, int r0, int r1, int r2, int sym,
                  double* norm_out, double* alpha_out, void* small_ws, void* stream);
/* Same for SFTuckerAdam (src/model/symmetric/optim.py:110-167): adam = device state
 * [v, ratio_prev, step_t, beta1, beta2, eps, step_velocity, -] (fp64, updated in place); alpha_out becomes
 * (1 - beta1) / ratio and hyper[2] (the momentum coefficient rt_small_project reads) beta1 * ratio_prev / ratio,
 * ratio = (1 - beta1^e) sqrt(v / (1 - beta2^e)) + eps, e = step_t // step_velocity + 1 (optim.py:139-144).
 * The kept tangent is the step DIRECTION; the reference's momentum is ratio_prev times it (transport is linear). */
int rt_small_norm_adam(const float* dS_g, const double* gram_R, const double* gram_S, const double* gram_O,
                       double* hyper, double* adam, int r0, int r1, int r2, int sym,
                       double* norm_out, double* alpha_out, void* small_ws, void* stream);
/*
 * rt_small_project: projection of the previous direction (tangent at the OLD point) onto the
 * tangent space at the current point -- TuckerRiemannian.project at asymmetric/optim.py:86.
 *   in : core (current), core_old, dS_old, M_i = U_i^T [U_i_old | dV_i_old]  (fp64 [r_i, 2r_i])
 *   out: pS[r0,r1,r2] fp32; for each mode K_i (fp64 [2r_i, r_i]) and L_i = -M_i K_i (fp64 [r_i,r_i])
 *        so that pV_i = [U_old|dV_old] K_i + U_i L_i.   Outputs are pre-scaled by hyper[2] (beta).
 */
int rt_small_project(const float* core, const float* core_old, const float* dS_old,
                     const double* M_R, const double* M_S, const double* M_O,
                     const double* hyper, int r0, int r1, int r2, int sym,
                     float* pS_beta, double* K_R, double* K_S, double* K_O,
                     double* L_R, double* L_S, double* L_O, void* small_ws, void* stream);
/*
 * The same projection in two calls, for a step with momentum: the part that needs neither A_i nor hyper runs while
 * rt_small_prepare's factorisation does, on the SMs the factorisation leaves idle.  Outputs are bit-identical to
 * rt_small_prepare followed by rt_small_project.
 * rt_small_prepare_project: rt_small_prepare plus the head of the projection (the transport of dS_old and the
 *   products with the current core).  Its inputs must stay unchanged until rt_small_norm_project.
 * rt_small_norm_project: rt_small_norm (adam == NULL) or rt_small_norm_adam, then the tail of the projection in the
 *   same program: pS_beta, K_i and L_i exactly as rt_small_project returns them, with the beta that hyper[2] holds
 *   after the norm.  M_i must be the matrices given to rt_small_prepare_project.
 */
int rt_small_prepare_project(const float* core, const float* core_old, const float* dS_old,
                             const double* M_R, const double* M_S, const double* M_O,
                             int r0, int r1, int r2, int sym, void* small_ws, void* stream);
int rt_small_norm_project(const float* dS_g, const double* gram_R, const double* gram_S, const double* gram_O,
                          double* hyper, double* adam, const double* M_R, const double* M_S, const double* M_O,
                          int r0, int r1, int r2, int sym, double* norm_out, double* alpha_out,
                          float* pS_beta, double* K_R, double* K_S, double* K_O,
                          double* L_R, double* L_S, double* L_O, void* small_ws, void* stream);
/* dS_dir = alpha * dS_g + pS_beta (pS_beta may be NULL).  asymmetric/optim.py:92 (core part). */
int rt_core_axpby(const float* dS_g, const double* alpha_dev, const float* pS_beta, int count,
                  float* dS_dir, void* stream);
/*
 * rt_small_retract: the N-independent part of construct().round(rank) (asymmetric/optim.py:106-108):
 *   in : core, dS_dir, Gram_i = dV_dir_i^T dV_dir_i (fp64), hyper (lr)
 *   out: core_new fp32; Z1_i, Z2_i (fp64 [r_i,r_i]) with U_i_new = U_i Z1_i + dV_dir_i Z2_i;
 *        Mn_i (fp64 [r_i, 2 r_i], may be NULL) = U_i_new^T [U_i | dV_dir_i] = [Z1_i^T | Z2_i^T Gram_i]: the
 *        transport Grams the next rt_small_project needs, obtained without another N-sized pass
 *        (exact when U_i^T U_i = I and U_i^T dV_dir_i = 0).
 */
int rt_small_retract(const float* core, const float* dS_dir,
                     const double* gram_R, const double* gram_S, const double* gram_O,
                     const double* hyper, int r0, int r1, int r2, int sym,
                     float* core_new, double* Z1_R, double* Z2_R, double* Z1_S, double* Z2_S,
                     double* Z1_O, double* Z2_O, double* Mn_R, double* Mn_S, double* Mn_O,
                     void* small_ws, void* stream);

/*
 * rt_epoch_batch: assemble batch [lo, lo + B) of a device-resident epoch (csrc/epoch.cu): the items are
 * perm[lo + b] (int64, e.g. torch.randperm on the device: the shuffle of DataLoader(shuffle=True), train.py:227);
 * feat_all [Q, feat_cols] int32 are the (s, r[, o]) rows, (off_all [Q+1], idx_all) the CSR of their target lists
 * (what KG_dataset.__getitem__ builds densely, src/data/Dataset.py:42-53).  Outputs: feat_out [B, feat_cols],
 * off_out [B+1], idx_out [cap] (cap >= the largest possible batch; lists are truncated at cap).  No host sync.
 */
int rt_epoch_batch(const int64_t* perm, int lo, int B, const int* feat_all, int feat_cols, const int* off_all,
                   const int* idx_all, int* feat_out, int* off_out, int* idx_out, int cap, void* stream);

/* Symmetric eigen-decomposition (block Jacobi, fp64), exposed for testing:
 * A[n,n] (destroyed) -> eigenvalues w[n] descending, eigenvectors V[n,n] (columns). */
size_t rt_eigh_ws_bytes(int n);
int rt_eigh(double* A, int n, double* w, double* V, void* ws, void* stream);
/* Orthonormal basis Y[n, r] (row-major, fp64) of the dominant r-dimensional invariant subspace of the symmetric
 * positive semi-definite A[n, n] (not modified), by trace-correcting purification + Newton-Schulz polar iteration
 * on the fp64 tensor cores (csrc/subspace.cu): what Tucker.round / SFTucker.round need from the SVD of an
 * unfolding (asymmetric/optim.py:108, symmetric/optim.py:55,102).  info (device int[4], may be NULL) receives
 * the purification and Newton-Schulz iteration counts.  Exposed for testing; rt_small_retract uses it in batch. */
size_t rt_dominant_subspace_ws_bytes(int n, int r);
int rt_dominant_subspace(const double* A, int n, int r, double* Y, int* info, void* ws, void* stream);

/* ---- (e) rank change ------------------------------------------------------------------- */
/*
 * rt_fill_normal: out[rows, cols] (row-major, dense) <- standard normal fp32 values, counter-based (csrc/fill.cu:
 * Philox4x32-10, Box-Muller).  The value at (row, col) depends only on (seed, stream_id, row_begin + row, col): a
 * shard that passes its first global row as row_begin draws exactly those rows of the draw over all rows, and every
 * caller that passes the same arguments gets the same bits.  stream_id separates independent draws under one seed.
 * Used by set_rank (rank.py) for the new factor directions and core entries of a rank increase.  rows == 0 or
 * cols == 0 launches nothing.
 */
int rt_fill_normal(float* out, int rows, int cols, int64_t row_begin, uint64_t seed, uint32_t stream_id,
                   void* stream);


#ifdef __cplusplus
}
#endif
#endif /* RTUCKER_H_ */
