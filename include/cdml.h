/* libcdml.so -- C ABI of the B200-native CDML hot path.
 *
 * The reference (geekieo/collaborative-deep-metric-learning) has no FFI of its own: its hot path is
 * Python calling TensorFlow 1.13 and faiss 1.5 ops.  Each entry point below replaces the library op(s)
 * the reference reaches at the cited call site (file:line relative to the reference tree) and is what a
 * ctypes binding in the reference's own modules would bind (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; cdml_last_error() gives the thread-local message;
 *   - no exceptions, no ownership transfer: all tensors are caller-owned DEVICE pointers unless a
 *     parameter is documented as host; row-major, explicit leading dimensions in ELEMENTS;
 *   - every compute call takes a cudaStream_t (as void*) and is asynchronous w.r.t. the host;
 *   - dtype16: 0 = fp16, 1 = bf16 (operand type of the tensor-core GEMMs; accumulation is fp32);
 *   - 16-bit / fp32 matrices handed to GEMMs need 16-byte aligned bases and row pitches.
 *
 * Collectives (deliberate deviation from SURVEY.md 8(b)'s draft list): there is NO cdml_nccl_init / cdml_allreduce_sum /
 * cdml_allgather.  The exchange steps of the path -- the all-reduce of the flat gradient buffer, the all-reduce MAX of the
 * per-query KNN bound pairs, the all-to-all of the per-shard KNN records -- are issued by the host through
 * torch.distributed (NCCL): the task assigns that plumbing to torch ("one process per GPU with torch.distributed over
 * NCCL/NVLink"), a second communicator inside this library would duplicate the process group's rendezvous, and NCCL calls
 * made by torch are what CUDA-graph capture of the whole training step records.  Every entry point that sits next to a
 * collective is shaped for it: contiguous flat buffers ([dW ; db] per layer, fp32 [2,nq] pairs, [nq,k] 64-bit records),
 * stream-ordered, no host synchronisation between the call and the collective.
 */
#ifndef CDML_H_
#define CDML_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cdml_ctx cdml_ctx;

#define CDML_F16 0
#define CDML_BF16 1

/* ---- context / errors ------------------------------------------------------------------------ */
int cdml_ctx_create(int device, cdml_ctx** out);
int cdml_ctx_destroy(cdml_ctx* ctx);
const char* cdml_last_error(void);
int cdml_version(void);
/* Device-side error word (bad gather index ...): copies it to *flags (host) and clears it. Synchronises stream. */
int cdml_ctx_poll_errors(cdml_ctx* ctx, void* stream, int32_t* flags);

/* ---- K1: triplet row gather -- replaces numpy FEATURES[np.asarray(guid_triplets)] (inputs.py:158) + reshape
 *      (train.py:313).  Bit-exact byte copy of n_idx rows of row_bytes each.  idx_is_64: int64 vs int32 indices;
 *      negative indices wrap like numpy; out-of-range sets error flag bit 0 and writes zeros. */
int cdml_gather_rows(cdml_ctx* ctx, const void* table, int64_t num_rows, int64_t row_bytes, int64_t table_pitch_bytes,
                     const void* idx, int idx_is_64, int64_t n_idx, void* out, int64_t out_pitch_bytes, void* stream);

/* ---- K2: row L2-normalise + cast -- replaces tf.nn.l2_normalize(model_input) (models.py:58) and the
 *      numpy row normalisation of calc_knn (faiss_knn.py:99-104).  in fp32 [n,F] -> out16 [n,ld_out] (columns
 *      F..ld_out-1 zeroed).  normalize: 0 = cast only, 1 = x*rsqrt(max(sum x^2,eps)) (TF), 2 = x/sqrt(sum x^2) (numpy).
 *      out32 (nullable) receives the fp32 normalised rows [n,ld_out32]; sumsq (nullable) the row sum of squares
 *      of the OUTPUT16 rows (after rounding) as fp32 [n]. */
int cdml_rows_normalize_cast(cdml_ctx* ctx, const float* in, int64_t n, int64_t F, int64_t ld_in, int normalize,
                             float eps, void* out16, int64_t ld_out, int dtype16, float* out32, int64_t ld_out32,
                             float* sumsq, void* stream);

/* ---- K3/K4/K6: tensor-core GEMM family (tcgen05 + TMA).  Replaces slim.fully_connected's MatMul/BiasAdd/
 *      LeakyRelu (models.py:26-30), tf.nn.l2_normalize(layer_2) (models.py:61) and the autodiff MatMuls of
 *      optimizer.compute_gradients (train.py:141-142).
 *      A is [M,K] (a_mn_major=0) or [K,M] (a_mn_major=1); B is [N,K] (b_mn_major=0) or [K,N] (b_mn_major=1).
 *      epilogue:
 *        0 STORE_F32  out fp32 [M,ld_out] = leaky(acc + bias)         (bias nullable; alpha=1 -> identity);
 *                     num_splits > 1 writes split-K partials at out + s*split_stride (reduce with cdml_sum_partials)
 *        1 STORE_16   out 16-bit [M,ld_out] = leaky(acc + bias); aux0 (nullable) = packed SIGN MASK out, uint32
 *                     [ceil(N/32)][ld_aux1] (chunk-major, pitch ld_aux1 >= M words): bit j of word [c][m] is set iff
 *                     acc + bias > 0 at column 32c+j -- all the backward pass needs of a leaky activation
 *        2 L2NORM     y = leaky(acc+bias); out fp32 = y*rsqrt(max(sum y^2,1e-12)); aux0 = rinv fp32 [M] (nullable);
 *                     aux1 = 16-bit copy [M,ld_aux1] (nullable).  Requires N <= 256.
 *        3 MASK_LEAKY out 16-bit = acc * (aux1[m,n] > 0 ? 1 : alpha)   (aux1 = 16-bit mask, ld_aux1)
 *        4 MASK_BITS  out 16-bit = acc * (bit ? 1 : alpha), aux1 = the packed sign mask a STORE_16 forward wrote
 *                     (same layout, pitch ld_aux1 words): the data gradient dz = (dy . W^T) * leaky'(z) of train.py:141-142
 *                     reading 1 bit instead of 16 per element
 *      num_splits: <=0 lets the library choose (STORE_F32 only); *splits_used (nullable, host) reports it. */
int cdml_gemm16(cdml_ctx* ctx, const void* A, int a_mn_major, int64_t lda, const void* B, int b_mn_major, int64_t ldb,
                int64_t M, int64_t N, int64_t K, int dtype16, int epilogue, void* out, int64_t ld_out,
                const float* bias, float alpha, void* aux0, void* aux1, int64_t ld_aux1, int num_splits,
                int64_t split_stride, int* splits_used, void* stream);
/* Split count the library would pick for (M,N,K) so callers can size the partial buffer. */
int cdml_gemm16_auto_splits(cdml_ctx* ctx, int64_t M, int64_t N, int64_t K);

/* out[i] = scale * sum_s parts[s*stride + i], fixed order (deterministic split-K / bias-grad reduction). */
int cdml_sum_partials(cdml_ctx* ctx, const float* parts, int num_parts, int64_t stride, int64_t n, float scale,
                      float* out, void* stream);

/* Column sums of a 16-bit matrix: out fp32 [N] = sum_rows X[r,:] (bias gradient of the autodiff, train.py:141).
 * workspace: fp32 [cdml_colsum_workspace_floats(R,N)]. */
int64_t cdml_colsum_workspace_floats(int64_t R, int64_t N);
int cdml_colsum16(cdml_ctx* ctx, const void* X, int64_t R, int64_t N, int64_t ld, int dtype16, float* workspace,
                  float* out, void* stream);

/* ---- K5: HingeLoss.calculate_loss (losses.py:21-49) forward + backward through the output L2-norm and the last
 *      leaky-ReLU.  E fp32 [3B,ld_e] rows a0,p0,n0,a1,...  neg_row (nullable int32 [B]) overrides the negative's row
 *      (in-batch mining); then gradients are scatter-added.  Outputs (all nullable except stats):
 *        pos_dist,neg_dist,hinge_dist fp32 [B]; stats fp32 [4] = {mean hinge (the loss), mean pos, mean neg, #active};
 *        dE fp32 [3B,ld_e] = d(sum_i hinge_i)/dE * grad_scale   (NOT divided by B unless grad_scale = 1/B);
 *        dz16 16-bit [3B,ld_dz] = (dE - e(e.dE)) * rinv * leaky'(e)  -- gradient w.r.t. the last layer's
 *        pre-activation, ready to be the A/B operand of the backward GEMMs.  rinv fp32 [3B] from the L2NORM epilogue.
 *      workspace: fp32 [3B*D] when dE is NULL but dz16 is requested. */
int cdml_triplet_hinge(cdml_ctx* ctx, const float* E, int64_t B, int D, int64_t ld_e, const int32_t* neg_row,
                       float margin, float grad_scale, const float* rinv, float leaky_alpha, float* pos_dist,
                       float* neg_dist, float* hinge_dist, float* stats, float* dE, void* dz16, int64_t ld_dz,
                       int dtype16, float* workspace, void* stream);

/* ---- K8: TF1 AdamOptimizer.apply_gradients (train.py:82,146) with exponential_decay (train.py:108-113).
 *      cdml_adam_prepare reads/increments the device step counter and writes lr_t (bias-corrected, decayed) to
 *      scalars[0] (device float[4]); cdml_adam_apply then updates one tensor and (optionally) its 16-bit shadow. */
int cdml_adam_prepare(cdml_ctx* ctx, int64_t* step_counter, float base_lr, float decay_steps, float decay_rate,
                      int staircase, float beta1, float beta2, float* scalars, void* stream);
int cdml_adam_apply(cdml_ctx* ctx, float* w, float* m, float* v, const float* g, int64_t n, const float* scalars,
                    float beta1, float beta2, float eps, float grad_scale, void* w16, int dtype16, void* stream);
/* ---- the rest of build_graph's gradient path (train.py:133-146) and its other optimizers.
 *      g_eff = grad_scale*g + wd_reg*w  (wd_reg = regularization_penalty * l2_penalty of slim.l2_regularizer, weights only);
 *      per-variable tf.clip_by_norm (train.py:47-64): g_eff *= clip_norm / max(||g_eff||, clip_norm) when clip_norm > 0;
 *      kind 0 Adam, 1 MomentumOptimizer(momentum, use_nesterov=True) (train.py:115-116),
 *           2 tf.contrib.opt.LARSOptimizer (train.py:354: trust = eeta*||w|| / (||g|| + wd*||w|| + eps) when both norms > 0,
 *             acc = momentum*acc + g, w -= lr*trust*acc -- TF r1.13's apply_momentum(var, mom, lr*trust, grad, momentum): the
 *             weight decay enters the trust ratio only), 3 GradientDescent.
 *      cdml_opt_sumsq writes out2 = {sum g_eff^2, sum w^2} for one variable (deterministic two-stage reduction;
 *      workspace fp32 [cdml_opt_workspace_floats()]); cdml_opt_apply reads them as `norms` (needed for clipping and
 *      LARS, NULL otherwise).  scalars = cdml_adam_prepare's output ([0] bias-corrected Adam step size, [1] decayed lr). */
int64_t cdml_opt_workspace_floats(void);
int cdml_opt_sumsq(cdml_ctx* ctx, const float* g, const float* w, int64_t n, float grad_scale, float wd_reg,
                   float* workspace, float* out2, void* stream);
int cdml_opt_apply(cdml_ctx* ctx, int kind, float* w, float* m, float* v, const float* g, int64_t n, const float* scalars,
                   const float* norms, float beta1, float beta2, float eps, float grad_scale, float wd_reg, float clip_norm,
                   float momentum, float lars_weight_decay, float lars_eeta, void* w16, int dtype16, void* stream);
/* ---- fusion towers (models.py:65-157): elementwise joins of 16-bit [rows, cols] activations (tf.multiply, the residual
 *      adds and their backward forms) and tf.nn.l2_normalize of a tensor that is not a GEMM output.
 *      op: 0 a*b | 1 a+b | 2 a*b+a+b | 3 a*leaky'(b) | 4 a*b+a | 5 a*b+c | 6 (a*b+a)*leaky'(c) |
 *      7 a*b*leaky'(c), leaky'(t) = t > 0 ? 1 : alpha; c may be NULL for ops < 5; cols and all pitches even. */
int cdml_ew16(cdml_ctx* ctx, int op, const void* a, int64_t lda, const void* b, int64_t ldb, const void* c, int64_t ldc,
              void* out, int64_t ldo, int64_t rows, int cols, float alpha, int dtype16, void* stream);
int cdml_rows_l2norm16(cdml_ctx* ctx, const void* y16, int64_t n, int D, int64_t ld_y, float eps, int dtype16, float* e,
                       int64_t ld_e, float* rinv, void* e16, int64_t ld_e16, void* stream);
/* fp32 -> 16-bit cast of a flat buffer (initial shadow weights). */
int cdml_cast16(cdml_ctx* ctx, const float* in, int64_t n, void* out16, int dtype16, void* stream);

/* X16[r, col] = value for every row r (16-bit matrix, pitch ld elements).  Used to plant the column of ones that turns
 * the bias gradient db = sum_rows dz (train.py:141) into one extra output row of the weight-gradient GEMM:
 * [x | 1]^T . dz = [dW ; db]. */
int cdml_fill_column16(cdml_ctx* ctx, void* X16, int64_t rows, int64_t ld, int64_t col, float value, int dtype16,
                       void* stream);

/* ---- row M: in-batch semi-hard negative mining (build-defined; SURVEY.md 8a row M).  E16 16-bit [3B,ld] embeddings,
 *      E32 fp32 [3B,ld32] (for |a-p|^2), guid int64 [B,3].  neg_row int32 [B] out, d_an fp32 [B] out (nullable). */
int cdml_mine_semihard(cdml_ctx* ctx, const void* E16, int64_t ld16, int dtype16, const float* E32, int64_t ld32,
                       const int64_t* guid, int64_t B, int D, float margin, int32_t* neg_row, float* d_an,
                       void* stream);
/* Distance-weighted negative sampling (Wu et al. 2017), the second mining mode: the same candidates and arguments as
 * cdml_mine_semihard, but the negative is SAMPLED among the candidates with max(d, cutoff^2) < dp + margin, with
 * probability proportional to the inverse density of squared distances on the unit sphere in D dimensions (the exact
 * definition and draw layout are stated in csrc/mine.cu and oracle/mine_dw_oracle.py).  Draws are keyed by (seed, *step,
 * anchor, chunk); step is a device pointer to an int64 read by the kernel (NULL: step 0), so a replayed CUDA graph draws
 * afresh at every step.  No eligible candidate: row 3i+2. */
int cdml_mine_distance_weighted(cdml_ctx* ctx, const void* E16, int64_t ld16, int dtype16, const float* E32,
                                int64_t ld32, const int64_t* guid, int64_t B, int D, float margin, float cutoff,
                                uint64_t seed, const int64_t* step, int32_t* neg_row, float* d_an, void* stream);
/* Diagnostics of the last cdml_mine_semihard or cdml_mine_distance_weighted on this context (synchronises `stream`): out2[0] = (anchor, 32-candidate
 * chunk) pairs the selection epilogue had to re-scan, out2[1] = anchors that received a mined negative. */
int cdml_mine_last_stats(cdml_ctx* ctx, int64_t* out2, void* stream);

/* ---- K11-K13: exact flat KNN -- replaces faiss index.add + index.search (faiss_knn.py:116-128) with
 *      IndexFlatL2 / IndexFlatIP semantics.  X fp32 [N,d] (ldx), Q fp32 [nq,d] (ldq); metric 0 = L2 (squared,
 *      ascending), 1 = IP (descending).  D fp32 [nq,k], I int64 [nq,k] (+id_offset; -1/inf padding when N < k).
 *      Workspace is internal to the index object.  The tensor-core pass only nominates candidates; the reported
 *      distances/order come from an exact fp32 re-rank (||q||^2+||x||^2-2q.x, clamped at 0 like faiss). */
typedef struct cdml_index cdml_index;
int cdml_knn_index_build(cdml_ctx* ctx, const float* X, int64_t N, int d, int64_t ldx, int metric, void* stream,
                         cdml_index** out);
int cdml_knn_index_destroy(cdml_index* index);
int cdml_knn_search(cdml_ctx* ctx, cdml_index* index, const float* Q, int64_t nq, int64_t ldq, int k, float* D,
                    int64_t* I, int64_t id_offset, void* stream);
/* Row-sharded index, two-phase search (the exchange between the phases is the caller's: NCCL all-reduce MAX of bound_full
 * and MIN of bound_part over the shards).  cdml_knn_bounds runs the bound pass only and writes, per query, the raw
 * k_full-th and k_part-th best sampled scores of THIS shard (-inf when the shard has no usable sample).  Any shard has
 * k_full rows above its bound_full, and every shard has k_part rows above the smallest bound_part, so with
 * k_part = ceil(k / shards) both max_s(bound_full) and min_s(bound_part) are lower bounds of the global k-th best score.
 * cdml_knn_search_bounded then collects only rows scoring above max(bound_full, bound_part) - slack: the shards together
 * nominate about as many candidates as one unsharded index instead of `shards` times as many. */
int cdml_knn_bounds(cdml_ctx* ctx, cdml_index* index, const float* Q, int64_t nq, int64_t ldq, int k_full, int k_part,
                    float* bound_full, float* bound_part, void* stream);
int cdml_knn_search_bounded(cdml_ctx* ctx, cdml_index* index, const float* Q, int64_t nq, int64_t ldq, int k,
                            const float* bound_full, const float* bound_part, float* D, int64_t* I, int64_t id_offset,
                            void* stream);
/* Counters of the last search: stats[0] = candidates nominated, [1] = queries that overflowed to the exact fallback. */
int cdml_knn_last_stats(cdml_index* index, int64_t* stats);
/* Merge G per-shard results [G,nq,k] into the global top-k (ties -> lower id). */
int cdml_knn_merge(cdml_ctx* ctx, const float* Dg, const int64_t* Ig, int G, int64_t nq, int k, int metric, float* D,
                   int64_t* I, void* stream);

/* Row-sharded index, protocol with ONE collective per phase (faiss_knn.sharded_search; the three calls process one chunk of
 * at most 65536 queries and share the index workspace, so they must follow each other on one stream):
 *   cdml_knn_shard_bounds   pair[0][q] = k-th best sampled score of this shard, pair[1][q] = -(k_part-th best)  (-inf / +inf
 *                           without a usable sample)                                       -> caller: all-reduce MAX of pair
 *   cdml_knn_shard_collect  collects the rows above max(pair[0], -pair[1]) - slack and writes nom_pair[0][q] = k-th best
 *                           approximate score among this shard's nominees, nom_pair[1][q] = -(k_part-th best)
 *                                                                                          -> caller: all-reduce MAX of nom_pair
 *   cdml_knn_shard_refine   exact fp32 re-rank of the nominees within 2*eps of max(nom_pair[0], -nom_pair[1]) -- a lower bound
 *                           of the GLOBAL k-th best approximate score, so the shards together re-rank ~k rows per query, not
 *                           shards*k -- and writes this shard's (possibly shorter than k) sorted list as 64-bit records
 *                           rec[q][j] = (order-preserving distance key << 32) | global id, padding = ~0
 *                                                                                          -> caller: all-to-all of rec
 *                           overflow_flag NULL: synchronises the stream and redoes queries whose candidate list overflowed
 *                           exactly (like cdml_knn_search).  Non-NULL (device int32): NO host synchronisation -- the word is
 *                           set to 1 if any query overflowed and the caller, after its exchange, repeats the search with
 *                           NULL in that (rare) case; the common case runs the whole protocol without a host round trip
 *   cdml_knn_merge_packed   k-way merge of G <= 32 record lists [G,nq,k] -> D, I [nq,k] (ties -> lower id), or -- rec_out
 *                           non-NULL -- the merged list as records [nq,k] (the caller all-gathers ONE 8-byte array and
 *                           cdml_knn_unpack_records turns records into D fp32 / I int64).
 * pair / nom_pair are fp32 [2,nq]; global ids (id_offset + row) must fit 32 bits. */
int cdml_knn_shard_bounds(cdml_ctx* ctx, cdml_index* index, const float* Q, int64_t nq, int64_t ldq, int k, int k_part,
                          float* pair, void* stream);
int cdml_knn_shard_collect(cdml_ctx* ctx, cdml_index* index, const float* Q, int64_t nq, int64_t ldq, int k, int k_part,
                           const float* pair, float* nom_pair, void* stream);
int cdml_knn_shard_refine(cdml_ctx* ctx, cdml_index* index, const float* Q, int64_t nq, int64_t ldq, int k,
                          const float* nom_pair, unsigned long long* rec, int64_t id_offset, int32_t* overflow_flag,
                          void* stream);
int cdml_knn_merge_packed(cdml_ctx* ctx, const unsigned long long* rec, int G, int64_t nq, int k, int metric, float* D,
                          int64_t* I, unsigned long long* rec_out, void* stream);
int cdml_knn_unpack_records(cdml_ctx* ctx, const unsigned long long* rec, int64_t n, int metric, float* D, int64_t* I,
                            void* stream);

/* ---- evaluate.Evaluation.mean_dist (evaluate.py:57-73): mean_p sum_d (V[p0]-V[p1])^2, pairs int64 [P,2]. */
int cdml_mean_pair_dist(cdml_ctx* ctx, const float* V, int64_t ld, int D, const int64_t* pairs, int64_t P,
                        float* out_mean, void* stream);

/* ---- de-similarity post-filter of the KNN lists -- replaces faiss_knn.iter_desim_mp (faiss_knn.py:187-244: fliter_fI,
 *      add_invalid_row, 81 x Pool(22) column sweeps of desim_progress) and faiss_knn.desim (faiss_knn.py:134-143).
 *      eI [n,ke] int64 embedding-KNN ids (-1 = padding), fI / fD [nf,kf] the raw-feature KNN (ids int64, squared distances
 *      fp32; fD may be NULL = no distance filter).  Per row, left to right: an entry still alive is a pivot v; every LATER
 *      entry found among v's first min(kf,f_end) feature neighbours (those with fD <= threshold, other than v itself) is
 *      dropped; finally the row's own id (row + row_offset: eI may be a slice of the rows, one slice per rank) is
 *      dropped.  out [n,ke] int64 = eI with dropped entries -1 (may alias eI).
 *      workspace: cdml_desim_workspace_bytes(nf,kf,f_end) device bytes.  ke <= 256, min(kf,f_end) <= 64, nf < 2^31.
 *      An id >= nf (IndexError in the reference) is left untouched and sets error flag bit 1 (cdml_ctx_poll_errors). */
int64_t cdml_desim_workspace_bytes(int64_t nf, int kf, int f_end);
int cdml_desim(cdml_ctx* ctx, const int64_t* eI, int64_t n, int ke, int64_t ld_e, const int64_t* fI, const float* fD,
               int64_t nf, int kf, int64_t ld_fi, int64_t ld_fd, float fD_threshold, int f_end, void* workspace,
               int64_t* out, int64_t ld_out, int64_t row_offset, void* stream);
/* out[i,j] = -1 where eI[i,j] occurs in fI[i,:], else eI[i,j]  (faiss_knn.desim). */
int cdml_desim_simple(cdml_ctx* ctx, const int64_t* eI, int64_t n, int ke, int64_t ld_e, const int64_t* fI, int kf,
                      int64_t ld_f, int64_t* out, int64_t ld_out, void* stream);

/* ---- on-device triplet reader -- replaces MPTripletPipe.subprocess + parse_data.yield_negative_index (inputs.py:102-142,
 *      parse_data.py:292-298) for a *.train file whose pairs [n_pairs,2] int64 are resident on the device.
 *      out[i] = (a, p, n), (a,p) = pairs[(start+i) % n_pairs], n uniform in [0,num_guid) re-drawn while n in {a,p}.
 *      Generator: Philox4x32-10, key = seed, counter = (start+i, attempt); Lemire multiply-shift with rejection. */
int cdml_sample_triplets(cdml_ctx* ctx, const int64_t* pairs, int64_t n_pairs, int64_t start, int64_t B, int64_t num_guid,
                         uint64_t seed, int64_t* out, void* stream);

/* ---- host-side text formats either side of the path (HOST pointers, no device work) ---------------------------------
 * cdml_format_knn_rows: the line format of faiss_knn.write_process (faiss_knn.py:267-283) for rows [begin_index,
 *      begin_index+nq): '<guid[q]>,' then for columns 1..k-1 with I > 0 and 0 < D < 1.4: '<guid[I]>#<str(np.float32(D))><',
 *      then '\n'.  guid_blob / guid_off [n_guids+1]: the decode map as one UTF-8 blob + offsets.  Returns the number of
 *      bytes written to out (capacity cap), or -1.
 * cdml_format_f32: str(numpy.float32(v)) + '\n' per value (the float formatting used above, exposed for tests).
 * cdml_parse_features_txt: online_data.read_features_txt (online_data.py:48-84) over a whole file image: every line
 *      'guid#f1,...,f<width>' whose fields parse as Python float() does (text -> double -> float32) becomes a row of out
 *      [max_rows,width] (max_rows >= number of lines), kept rows compacted to the front in file order; guid_begin /
 *      guid_len give each kept row's guid as a slice of buf.  Lines without exactly one '#', with an unparsable field or
 *      with another field count are dropped.  Returns the number of kept rows, or -1. */
int64_t cdml_format_knn_rows(const float* D, const int64_t* I, int64_t nq, int k, int64_t ld, int64_t begin_index,
                             const char* guid_blob, const int64_t* guid_off, int64_t n_guids, char* out, int64_t cap);
int64_t cdml_format_f32(const float* v, int64_t n, char* out, int64_t cap);
int64_t cdml_parse_features_txt(const char* buf, int64_t len, int width, float* out, int64_t max_rows, int64_t* guid_begin,
                                int32_t* guid_len, int num_threads);

#ifdef __cplusplus
}
#endif
#endif /* CDML_H_ */
