/* yue_b200.h -- C ABI of the B200-native BPR hot path (libyue_b200.so).
 *
 * The reference (0411tony/Yue) is pure Python and has NO FFI of its own; this is the thin
 * boundary a maintainer binds with ctypes from recommender/cf/BPR.py (see INTEGRATION.md).
 * Each entry point names the reference code it replaces (paths relative to the reference
 * tree).  Conventions: every function returns 0 on success or a YUE_E_* code, with a
 * message available from yue_last_error(); the caller owns every host buffer, the library
 * owns every device buffer; no global mutable state; one host thread per handle, distinct
 * handles are independent; plain pointers and sizes only.
 *
 * Array form of the play log (built from data/record.py's Record by the host side):
 *   ev_indptr[m+1] int64, ev_items[T] int32   every training event, user-major in user-id
 *        order (= first-appearance order, recommender/cf/BPR.py:42), file order inside a
 *        user, repeat plays kept (BPR.py:44-45).  One BPR triplet per event.
 *   uq_indptr[m+1] int64, uq_items[nnz] int32  per-user SORTED UNIQUE played tracks
 *        (= userListen, BPR.py:32-35): the sampler's rejection set and the ranking mask
 *        (base/IterativeRecommender.py:102-106).
 * Factor tables are dense row-major float32, P[m,k] and Q[n,k]
 * (base/IterativeRecommender.py:36-39).
 */
#ifndef YUE_B200_H
#define YUE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct yue_handle yue_t;

enum {
    YUE_OK = 0,
    YUE_E_ARG = 1,      /* bad argument / call order                                  */
    YUE_E_CUDA = 2,     /* CUDA runtime error (message has the cudaError string)      */
    YUE_E_STATE = 3,    /* interactions or factors not set                            */
    YUE_E_NUMERIC = 4,  /* loss is NaN or infinite (IterativeRecommender.py:63-66)    */
    YUE_E_NCCL = 5,
    YUE_E_UNSUPPORTED = 6
};

/* update schedule of yue_bpr_epoch / yue_bpr_apply */
enum {
    YUE_MODE_SERIAL = 0,        /* one warp, events strictly in order: reproduces the
                                   reference loop given the same negatives (parity mode) */
    YUE_MODE_HOGWILD = 1,       /* throughput mode: warps pull users from a cursor in stream
                                   order, a user's triplets stay in order inside a warp, row
                                   changes are published as vector atomic deltas          */
    YUE_MODE_HOGWILD_STORE = 2  /* as HOGWILD but plain stores (last writer wins)         */
};

/* algorithm of yue_rank_topn */
enum {
    YUE_RANK_EXACT = 0,   /* fp32 FMA-chain scores on CUDA cores, fused masked top-N      */
    YUE_RANK_TC = 1,      /* tcgen05 tf32 candidate pass + exact fp32 re-score (same ids) */
    YUE_RANK_AUTO = 2
};

/* which device buffer yue_device_buffer exposes (for torch.distributed plumbing) */
enum { YUE_BUF_P = 0, YUE_BUF_Q = 1, YUE_BUF_Q_DELTA = 2, YUE_BUF_Q_SNAPSHOT = 3 };

const char* yue_version(void);
const char* yue_last_error(const yue_t* h);          /* h may be NULL: last create error */

/* Number of CUDA devices (0 without a driver).  The host driver maps `-cv k -p` folds onto devices with it, where
 * the reference runs the folds as processes and divides MKL threads among them (yue.py:72-105). */
int yue_device_count(int* count);
int yue_create(int device, yue_t** out);
int yue_destroy(yue_t* h);
int yue_sync(yue_t* h);

/* pinned host memory, so the P/Q/ids arrays the Python class exposes can be DMA targets */
int yue_host_alloc(size_t bytes, void** out);
int yue_host_free(void* p);

/* Replaces the userListen build and the epoch iteration order, BPR.py:32-45 (id-keyed
 * variant BPR.py:84-91).  The shard form is for user-sharded multi-GPU runs: this handle
 * owns users [user_begin, user_begin + m_local); event_base is the global index of its first
 * event (the sampler stream is a function of the GLOBAL event index, so samples do not
 * depend on the sharding).  yue_set_interactions == shard with user_begin = event_base = 0. */
int yue_set_interactions(yue_t* h, int64_t m, int64_t n,
                         const int64_t* ev_indptr, const int32_t* ev_items,
                         const int64_t* uq_indptr, const int32_t* uq_items);
int yue_set_interactions_shard(yue_t* h, int64_t m_local, int64_t n,
                               int64_t user_begin, int64_t event_base,
                               const int64_t* ev_indptr, const int32_t* ev_items,
                               const int64_t* uq_indptr, const int32_t* uq_items);

/* For shards that are not a contiguous range of users (yue_b200/sharding.py: interleaved_users): per local user,
 * the offset that turns a local event index into the global one (global = local + delta[user]); replaces the
 * single event_base of yue_set_interactions_shard so that the sampler stream stays that of the unsharded log.
 * NULL switches back to event_base.  Reset by the next yue_set_interactions. */
int yue_set_event_offsets(yue_t* h, const int64_t* delta);

/* Builds the same arrays ON THE DEVICE from the events in file order (SURVEY.md 8f row 1): replaces the
 * array-building half of Record.preprocess (data/record.py:138-202: userRecord grouping 147-165,
 * testSet with the training pairs removed 182-202) and BPR.py:32-45 for logs whose users and tracks are
 * already numbered (ids by first appearance stay with the host, record.py:138-146).  ev_user[E],
 * ev_item[E] in file order, is_test[E] != 0 marks held-out events (NULL: none).  Afterwards the handle is
 * in the state yue_set_interactions + yue_set_test_set would leave it in; the getters return the arrays
 * (sizes from yue_interaction_sizes; any pointer may be NULL). */
int yue_ingest_events(yue_t* h, int64_t m, int64_t n, int64_t E, const int32_t* ev_user,
                      const int32_t* ev_item, const uint8_t* is_test);
int yue_interaction_sizes(yue_t* h, int64_t* m, int64_t* n, int64_t* T, int64_t* nnz, int64_t* n_test);
int yue_get_interactions(yue_t* h, int64_t* ev_indptr, int32_t* ev_items, int64_t* uq_indptr, int32_t* uq_items);
int yue_get_test_set(yue_t* h, int64_t* test_indptr, int32_t* test_items);

/* Replaces IterativeRecommender.initModel's tables (IterativeRecommender.py:36-39) on the
 * device: P is [m_local,k], Q is [n,k].  get copies the current tables back (either pointer
 * may be NULL) -- buildModel leaves self.P / self.Q on the host (BPR.py:127-128). */
int yue_set_factors(yue_t* h, int k, const float* P, const float* Q);
int yue_get_factors(yue_t* h, float* P, float* Q);

/* Replaces `choice(itemList)` + redraw-while-played, BPR.py:46-49 (BPR.py:73-76,
 * recommender/advanced/APR.py:104-107).  Writes the accepted negative of every local event
 * for (seed, epoch, slot); bit-exact with oracle/philox.py.  Check hook: the epoch kernels
 * sample in-register and never materialise this array. */
int yue_sample_negatives(yue_t* h, uint64_t seed, uint32_t epoch, uint32_t slot,
                         int32_t* j_out);

/* Replaces one pass of the SGD loop body, BPR.py:42-58, over every local event, negatives
 * drawn in-kernel.  *loss_out (may be NULL: no host sync) receives sum of -log(s), BPR.py:58;
 * the caller adds regU*|P|^2 + regI*|Q|^2 from yue_frob2 (BPR.py:59) and runs the lr
 * schedule (IterativeRecommender.py:47-75) on the host. */
int yue_bpr_epoch(yue_t* h, double lr, double regU, double regI,
                  uint64_t seed, uint32_t epoch, int mode, double* loss_out);

/* One SUB-EPOCH: the part-th of n_parts consecutive ranges of the epoch's work (users in stream order).
 * Running part = 0..n_parts-1 in turn is the epoch; the multi-GPU trainer reconciles Q between parts
 * (SURVEY.md 8e: one all-reduce of the Q deltas per sub-epoch).  *loss_out is the part's share. */
int yue_bpr_epoch_part(yue_t* h, double lr, double regU, double regI,
                       uint64_t seed, uint32_t epoch, int mode, int part, int n_parts, double* loss_out);

/* Same update on a caller-supplied triplet stream (parity hook for the "same triplet
 * stream" check of north_star; also the building block for APR-style batches). */
int yue_bpr_apply(yue_t* h, const int32_t* u, const int32_t* i, const int32_t* j, int64_t T,
                  double lr, double regU, double regI, int mode, double* loss_out);

/* APR (adversarial BPR, recommender/advanced/APR.py:25-76, config C5): the same pass with the
 * adversarial perturbation fused per triplet -- loss softplus(-y) + regA softplus(-y_adv),
 * delta = eps * normalised gradient, held constant in the step (oracle/apr_ref.py states the
 * closed forms).  `slot` numbers the negative of each positive (the reference draws 3 per
 * positive, APR.py:95-111: call with slot = 0, 1, 2).  Replaces the body of APR.buildModel's
 * adversarial phase (APR.py:129-137); the first phase (APR.py:120-127) is yue_bpr_epoch. */
int yue_apr_epoch(yue_t* h, double lr, double regU, double regI, double eps, double regA,
                  uint64_t seed, uint32_t epoch, uint32_t slot, int mode, double* loss_out);
int yue_apr_apply(yue_t* h, const int32_t* u, const int32_t* i, const int32_t* j, int64_t T,
                  double lr, double regU, double regI, double eps, double regA, int mode,
                  double* loss_out);

/* CUNE's two-level BPR (recommender/advanced/CUNE.py:118-178; SURVEY.md 8f row 4).
 * yue_cune_set_implicit replaces the `implicit positive` sets CUNE.py:95-113 builds: ip_items[ip_indptr[u] ..
 * ip_indptr[u+1]) are the tracks of user u's top-K similar users that u has NOT played (a played track is refused,
 * YUE_E_ARG); m+1 / ip_indptr[m] entries, local user indices, copied to the device.  A new log drops them.
 * yue_cune_epoch replaces one pass of the training loop (CUNE.py:122-174): for every event (u, i), three repeats, each
 * drawing an implicit positive k (Philox slot 64 + repeat, attempt 0, position (r * len) >> 32 in the user's list) and
 * an unplayed track j (slot = repeat, rejection as in yue_bpr_epoch), then the ten row statements of CUNE.py:134-159
 * with every sigmoid re-evaluated on the current rows; users without implicit positives take the plain BPR step of
 * CUNE.py:164-171.  `s` is CUNE.conf's -s (> 0).  mode YUE_MODE_SERIAL reproduces the reference's order and rounding
 * (float32 rows, float64 scalars) and adds regU*|P|^2 + regI*|Q|^2 to the loss after EVERY user like CUNE.py:174;
 * YUE_MODE_HOGWILD runs one warp per user and adds (users with events) x the end-of-epoch norms instead.
 * *loss_out is the epoch's loss as CUNE.py:161-174 accumulates it; a non-finite loss is YUE_E_NUMERIC. */
int yue_cune_set_implicit(yue_t* h, const int64_t* ip_indptr, const int32_t* ip_items);
int yue_cune_epoch(yue_t* h, double lr, double regU, double regI, double s,
                   uint64_t seed, uint32_t epoch, int mode, double* loss_out);

/* LightGCN (recommender/advanced/LightGCN.py:15-105 on base/DeepRecommender:22-35; SURVEY.md 8f row 4).  The TF-1 graph:
 * e_0 = [U; V], e_k = A e_{k-1}, F = e_0 + sum_k l2_normalize(e_k) (37-45), A = one SparseTensor entry of value count(u, t)
 * per training EVENT and direction, duplicates summed, i.e. weight count^2 per pair (29-33: built here from the resident
 * log's play counts); loss = -sum log sigmoid(F_u.(F_i - F_j)) + reg/2 (|F_u|^2 + |F_i|^2 + |F_j|^2) over a batch (83-87);
 * AdamOptimizer(lr) on every row of U and V (88-90).  U, V are the handle's factor tables (yue_set_factors: the
 * truncated-normal init of DeepRecommender:30-31 is the caller's); a new yue_set_factors restarts Adam.
 * yue_gcn_set_events: the training events in FILE order -- next_batch_pairwise (56-79) walks `trainingData` in slices of
 *   batch_size; they must be the resident log's events (YUE_E_ARG otherwise).
 * yue_gcn_epoch: steps [step_begin, step_end) of one pass (step_end < 0: to the end; ceil(T / batch_size) steps per pass);
 *   step s trains on events [s * batch_size, ...), one negative per event: the FIFTH draw (Philox slot 4, event = file
 *   index, rejection against the user's plays) -- the reference draws five and keeps the last (68-78).
 *   loss_out[s - step_begin] = that step's loss (what line 97 prints).  All steps run in one cooperative launch.
 * yue_gcn_apply: one step on the caller's triplets (parity hook, no sampler).
 * yue_gcn_finalize: P, Q <- the propagated tables F (what predict() ranks with, 45-47 and 101-105), so that yue_predict /
 *   yue_rank_topn / yue_get_factors see them; the variables are kept and come back on the next yue_gcn_epoch / _apply. */
int yue_gcn_set_events(yue_t* h, int64_t T, const int32_t* ev_user, const int32_t* ev_item);
int yue_gcn_epoch(yue_t* h, int n_layers, int batch_size, double lr, double reg, uint64_t seed, uint32_t epoch,
                  int64_t step_begin, int64_t step_end, double* loss_out);
int yue_gcn_apply(yue_t* h, int n_layers, int64_t B, const int32_t* u, const int32_t* i, const int32_t* j,
                  double lr, double reg, double* loss_out);
int yue_gcn_finalize(yue_t* h, int n_layers);
/* Adam's state (checkpointing; tests read the first step's gradient from it: m_1 = 0.1 g): first / second moments of U and
 * V, [m, k] and [n, k] each (NULL = skip), and the number of steps taken since yue_set_factors. */
int yue_gcn_moments(yue_t* h, float* m_users, float* m_tracks, float* v_users, float* v_tracks, int64_t* steps);

/* BPR as the reference ships it (recommender/cf/BPR.py:65-129, SURVEY.md 3.3; the per-triplet loop of 31-62 is commented out
 * there): a TF-1 graph trained with AdamOptimizer on sampled mini-batches.  Step s draws `batch` training events uniformly
 * with replacement (next_batch, 65-81: np.random.randint at 66) and, per event, `negatives` unplayed tracks (uniform
 * over all n tracks, random.randint rejected against the user's plays, 74-76); loss = sum over the batch x negatives triplets of
 * softplus(-(U_u.V_i - U_u.V_j)) + reg (l2_loss(U_u) + l2_loss(V_i) + l2_loss(V_j)) with the rows read before the step
 * (93-115; regU for all three terms); one Adam step (beta 0.9 / 0.999, epsilon 1e-8) on EVERY row of U and V, num.max.iter steps (121-129).
 * U, V are the handle's factor tables (the graph's truncated_normal(0.005) init is the caller's); yue_set_factors restarts
 * Adam.  The moments are this path's own (not yue_gcn_*'s).  Sampler: Philox (yue_sample_negatives' stream) with epoch = s,
 * event = the batch row b: the event is attempt 0 of slot 4095 scaled to [0, T) (e = (r T) >> 32), negative k is slot k with
 * rejection -- the batch is a pure function of (seed, s).  Needs the whole log on one handle, T < 2^32, negatives <= 4095.
 * yue_bpr_adam_sample:  check hook (needs the log, not the factors), the batch of step `step`: events_out[batch]
 *   (indices into the event CSR) and neg_out[batch * negatives] (row-major by batch row).  Replaces next_batch, BPR.py:65-81.
 * yue_bpr_adam_steps:   steps [step_begin, step_end); loss_out[s - step_begin] = that step's loss (may be NULL), what
 *   the loop prints.  Replaces the loop of BPR.py:121-129 (the graph's Session.run).  Any split of a step range gives
 *   the same bits as the whole range; a non-finite loss is YUE_E_NUMERIC.
 * yue_bpr_adam_apply:   one step on the caller's B triplets (parity hook, no sampler); *loss_out = its loss.
 * yue_bpr_adam_moments: Adam's first / second moments of U and V ([m, k], [n, k]; NULL = skip) and the steps taken since
 *   yue_set_factors (checkpointing; tests read the first step's gradient from them: m_1 = 0.1 g). */
int yue_bpr_adam_sample(yue_t* h, uint64_t seed, int64_t step, int batch, int negatives, int32_t* events_out, int32_t* neg_out);
int yue_bpr_adam_steps(yue_t* h, int batch, int negatives, double lr, double reg, uint64_t seed, int64_t step_begin,
                       int64_t step_end, double* loss_out);
int yue_bpr_adam_apply(yue_t* h, int64_t B, const int32_t* u, const int32_t* i, const int32_t* j, double lr, double reg,
                       double* loss_out);
int yue_bpr_adam_moments(yue_t* h, float* m_users, float* m_tracks, float* v_users, float* v_tracks, int64_t* steps);

/* (P*P).sum(), (Q*Q).sum() of BPR.py:59, accumulated in float64. */
int yue_frob2(yue_t* h, double* p2, double* q2);

/* Replaces predict, BPR.py:131-134 / IterativeRecommender.py:58-60: scores[n] = Q.P[user]
 * as the canonical float32 FMA chain k = 0..d-1.  `user` is a local user index. */
int yue_predict(yue_t* h, int64_t user, float* scores_out);

/* Replaces the per-user body of evalRanking, IterativeRecommender.py:93-145: score every
 * track, drop the user's training tracks, keep the N best.  Output order is (score desc,
 * track id asc) -- exact top-N, see DESIGN.md for why the reference's lossy selection is not
 * reproduced.  ids_out/scores_out are [B,N]; rows with fewer than N unmasked tracks are
 * padded with -1 / -inf.  users[] are local user indices. */
int yue_rank_topn(yue_t* h, const int32_t* users, int64_t B, int N, int algo,
                  int32_t* ids_out, float* scores_out);

/* Replaces Measure.rankingMeasure, evaluation/measure.py:16-41 (hits 7-13, precision 51-53,
 * recall 91-94, MAP 56-66, coverage 43-48) plus the binary-relevance NDCG@n the reference lacks,
 * for the lists the last yue_rank_topn left on the device.  yue_set_test_set uploads Record.testSet
 * (data/record.py:195-202) as a CSR over the local users: test_indptr[m+1], test_items sorted unique
 * per user.  yue_rank_metrics: for each cut-off n = cuts[k] (the -topN list) sums_out[k*4 + {0,1,2,3}]
 * = sum over the ranked rows of {hits, hits/|test(u)|, AP, NDCG} and distinct_out[k] = number of
 * distinct tracks in the first n columns; the caller divides (precision = hits/(rows*n), recall =
 * sum/rows, MAP = sum/rows, coverage = distinct/itemCount).  Sums are reduced in a fixed order. */
int yue_set_test_set(yue_t* h, const int64_t* test_indptr, const int32_t* test_items);
int yue_rank_metrics(yue_t* h, int n_cuts, const int32_t* cuts, double* sums_out, int64_t* distinct_out);

/* The result lines of evalRanking, IterativeRecommender.py:145-155, for B ranked users at once (host code, all cores; no
 * device involved, no handle): line b = name of user b + ':' + for every id >= 0 of ids[b*N ..] the track's name, followed by
 * '*' where hits[b*N + r] != 0, + '\n'.  Names come as one byte blob per kind with offsets (name x = blob[off[x] .. off[x+1])):
 * user_off has B+1 entries (the B ranked users in order), track_off n_tracks+1.  The lines are written back to back into
 * out (out_cap bytes); *out_len = bytes needed -- when it exceeds out_cap nothing is written and YUE_E_ARG is returned, so a
 * first call with out = NULL, out_cap = 0 sizes the buffer.  With 1 M users x 10 tracks the reference's loop -- and a
 * column-wise numpy version of it -- take seconds; this takes a fraction of one. */
int yue_result_lines(const char* user_blob, const int64_t* user_off, const char* track_blob, const int64_t* track_off,
                     int64_t n_tracks, const int32_t* ids, const uint8_t* hits, int64_t B, int N,
                     char* out, int64_t out_cap, int64_t* out_len);

/* ---- WRMF (SURVEY.md 8f row 4: the next model on the same tables and the same ranking path) ----
 * One half-sweep of the implicit-feedback ALS of recommender/cf/WRMF.py (X = P table, Y = Q table of the handle):
 *   side 0  replaces the user loop, WRMF.py:34-57:  for every user  A = YtY + Y^T diag(alpha r_ui) Y + reg I,
 *           b = sum over played tracks of (1 + alpha r_ui) Y[i],  X[u] = inv(A) b   (float64, stored as float32);
 *           *loss_out (may be NULL) = sum over played pairs of (1 - X[u].Y[i])^2 with the X[u] from BEFORE the
 *           update, WRMF.py:49-50.
 *   side 1  replaces the track loop, WRMF.py:60-80, from the X just computed and listened[track][user].
 * r_ui = plays of track i by user u in the training log (WRMF.py:28-33), counted on the device from the event CSR;
 * alpha = 10 and reg = reg.lambda -u on BOTH sides in the reference (WRMF.py:55,79).  Users/tracks without training
 * plays get a zero row, as in the reference (b = 0).  num.factors <= 128.  The Gram matrix is accumulated in
 * float64 (the reference's YtY is a float32 sgemm): factors agree with the reference class to ~5e-6 per row.
 * Ranking afterwards is yue_rank_topn (predict = Y.dot(X[u]), WRMF.py:86-88). */
int yue_wrmf_sweep(yue_t* h, int side, double reg, double alpha, double* loss_out);
/* The same for rows [row_begin, row_end) only (*loss_out = their share).  Rows of a sweep are independent, so N
 * GPUs that hold the same log and tables each solve a range and exchange the solved rows (yue_b200/sharding.py:
 * WrmfShardedTrainer) -- the result is bit-identical to one GPU's. */
int yue_wrmf_sweep_rows(yue_t* h, int side, int64_t row_begin, int64_t row_end, double reg, double alpha, double* loss_out);
/* Check hook: the pair counts (aligned with uq_items) and the track-major form of the play sets the sweeps use
 * (it_indptr[n+1], it_users[nnz] sorted inside a track, it_counts[nnz]); any pointer may be NULL. */
int yue_wrmf_pair_counts(yue_t* h, int32_t* uq_counts, int64_t* it_indptr, int32_t* it_users, int32_t* it_counts);

/* ---- multi-GPU: user-sharded SGD with Q replicated; once per sub-epoch
 *      Q <- Q_snapshot + sum_over_ranks(Q_rank - Q_snapshot).  No reference counterpart
 *      (the reference has no collective anywhere, SURVEY.md section 2.1). ---- */
int yue_q_snapshot(yue_t* h);       /* snapshot <- Q                                        */
int yue_q_delta_pack(yue_t* h);     /* delta <- Q - snapshot                                */
int yue_q_delta_apply(yue_t* h);    /* Q <- snapshot + w * delta (after the reduction); snapshot <- Q */
/* Per-track factor w[n] applied to the summed deltas by yue_q_delta_apply / yue_allreduce_q_delta (NULL: 1).
 * The sum of the ranks' deltas overshoots for tracks played thousands of times between two exchanges (every
 * rank has already moved the row to its equilibrium); yue_b200/sharding.py: saturation_weights computes
 * (1 - a^G) / (G (1 - a)), a = exp(-kappa * plays per rank and exchange).  DESIGN.md section 6. */
int yue_set_delta_weights(yue_t* h, const float* w);
int yue_device_buffer(yue_t* h, int which, void** dev_ptr, size_t* bytes);   /* YUE_BUF_* */
int yue_stream(yue_t* h, void** cuda_stream);
/* NCCL path for non-Python hosts: id is an ncclUniqueId (128 bytes) from yue_comm_unique_id
 * on rank 0, distributed by the caller. */
int yue_comm_unique_id(void* id128);
int yue_comm_init(yue_t* h, int nranks, int rank, const void* id128);
int yue_allreduce_q_delta(yue_t* h);   /* pack + ncclAllReduce(sum, fp32) + apply            */

/* ---- multi-GPU, round 2: the most played tracks' rows live ONCE, the long tail is exchanged under the next sub-epoch ----
 * Why: summed deltas of a row that every rank touches thousands of times between two exchanges overshoot (every rank has
 * already made the whole move towards the row's equilibrium); profiles/quality_study_r1.md section E.  So the rows of
 * the hot tracks (the hot-row table of the blocked kernel, bpr_sgd_blk.cuh) are not replicated at all: slot s of the
 * table lives in the table of rank s % nranks, every rank maps every table (CUDA IPC between processes, plain peer
 * access inside one process) and the epoch kernel of every rank loads and adds (ld/red .sys) the one copy over NVLink.
 * All ranks must use the same hot set in the same slot order:
 *   yue_hot_tracks      the handle's current hot set (chosen from its own log by yue_set_interactions): tracks_out[n_hot]
 *   yue_set_hot_tracks  impose a hot set (tracks[] in slot order, counts[] = plays over ALL ranks, total_events likewise;
 *                       n_hot <= 248 -- the sharded trainer shares every track above 1/4096 of the events, one GPU's own
 *                       rule keeps the ~10 above 1/128; tracks above 1/40 get a second accumulator row); re-labels the events
 *   yue_hot_table_export / _open   this handle's table as a cudaIpcMemHandle_t (64 bytes) / map a peer's in this process
 *   yue_enable_peer     cudaDeviceEnablePeerAccess from the handle's device to `peer_device` (same-process handles)
 *   yue_hot_share       tables[r] = rank r's table as a device pointer valid in this process (tables[rank] may be NULL);
 *                       moves the rows this rank owns from Q into its table; from here on yue_bpr_epoch(_part) /
 *                       yue_apr_epoch(_part) in YUE_MODE_HOGWILD work on the shared tables and Q's hot rows are STALE.
 *                       Barrier between the ranks before the first epoch call.  After such an epoch yue_rank_topn,
 *                       yue_predict and yue_get_factors (with Q) return YUE_E_STATE until the next yue_hot_pull.
 *   yue_hot_pull        copy every hot row from its owner's table into this handle's Q (ranks quiescent: sync + barrier
 *                       before, barrier after if anyone goes on training)
 *   yue_hot_unshare     yue_hot_pull, then back to the per-launch private table
 * Needs num.factors = 32, 64 or 128 (the full-width blocked kernel). */
int yue_hot_tracks(yue_t* h, int32_t* tracks_out, int* n_hot);
int yue_set_hot_tracks(yue_t* h, const int32_t* tracks, const int64_t* counts, int n_hot, int64_t total_events);
int yue_hot_table_export(yue_t* h, void* ipc_handle64, void** dev_ptr);
int yue_hot_table_open(yue_t* h, const void* ipc_handle64, void** dev_ptr);
int yue_enable_peer(yue_t* h, int peer_device);
int yue_hot_share(yue_t* h, int nranks, int rank, void* const* tables);
int yue_hot_pull(yue_t* h);
int yue_hot_unshare(yue_t* h);
/* Exchange of the long tail, overlapped: begin packs delta = own = Q - snapshot on the handle's stream and lets its
 * SECOND stream (yue_stream2) wait for that; the caller all-reduces BUF_Q_DELTA on the second stream
 * (yue_q_exchange_reduce: the library's NCCL communicator; or torch.distributed on that stream) while the next sub-epoch
 * runs on the first; finish makes the first stream wait for the reduction and applies
 *     Q += w * sum - own,   snapshot += w * sum
 * i.e. the other ranks' changes arrive one sub-epoch late and this rank's own newer changes are kept.  quiescent != 0
 * states that no epoch ran on this handle since begin (the end of training): Q is then written as the new snapshot
 * itself, so that all ranks hold the same bits. */
int yue_q_exchange_begin(yue_t* h);
int yue_q_exchange_reduce(yue_t* h);
/* The reduction for ranks that are handles of ONE process (the class API with yue.devices=0,1,...; no NCCL involved):
 * deltas[r] = rank r's YUE_BUF_Q_DELTA (NULL = this handle's own), peer access enabled (yue_enable_peer).  Every rank
 * sums all ranks' deltas in rank order on its second stream and returns when that is done.  The caller synchronises:
 * every rank's yue_q_exchange_begin has completed (yue_sync + a barrier) before anyone calls this, and a barrier
 * after it before anyone's next yue_q_exchange_begin. */
int yue_q_exchange_reduce_peers(yue_t* h, int nranks, void* const* deltas);
int yue_q_exchange_finish(yue_t* h, int quiescent);
int yue_stream2(yue_t* h, void** cuda_stream);
/* Concurrency of the Hogwild epoch kernels: n_warps warps on n_ctas CTAs (one CTA per SM; 0 = the automatic choice of
 * yue_set_interactions).  With N ranks sharing the hot rows the number of updates of one row that are in flight between
 * a read and the add becoming visible grows N-fold plus the NVLink round trip; tools/staleness_sim.py and DESIGN.md
 * section 6 show where the trajectory leaves the 0.5-point gate.  Fewer CTAs than SMs also leave room for the NCCL
 * kernels of the overlapped exchange. */
int yue_set_sgd_concurrency(yue_t* h, int n_warps, int n_ctas);
/* yue_apr_epoch for the part-th of n_parts ranges of the work items (see yue_bpr_epoch_part) */
int yue_apr_epoch_part(yue_t* h, double lr, double regU, double regI, double eps, double regA, uint64_t seed,
                       uint32_t epoch, uint32_t slot, int mode, int part, int n_parts, double* loss_out);

/* ---- measurement hooks (bench.py): CUDA events on the handle's stream, launch counter ---- */
int yue_timer_start(yue_t* h);
int yue_timer_stop(yue_t* h, float* ms);
int yue_launch_count(yue_t* h, int64_t* n);
/* diagnostics of the last yue_rank_topn that took the tcgen05 path: rows whose candidate buffer
 * spilled into the global pool, and rows that had to be redone by the exact kernel */
int yue_rank_stats(yue_t* h, int64_t* fallback_rows, int64_t* spilled_rows);
int yue_flush_l2(yue_t* h);            /* overwrite a >L2-sized scratch buffer              */

#ifdef __cplusplus
}
#endif
#endif /* YUE_B200_H */
