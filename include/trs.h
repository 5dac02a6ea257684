/* trs.h -- C ABI of libtrs_b200.so: the B200 (sm_100a) hot path of TorchRecSys.
 *
 * The reference (FrancescoI/torchrecsys) is pure Python on stock torch and has no FFI of its
 * own; every entry point below replaces a span of reference Python (cited per function,
 * paths relative to the reference root) and is what a binding for that span would call.
 * INTEGRATION.md shows the ctypes stubs.
 *
 * Rules of the boundary
 *  - plain C: pointers, sizes, PODs.  No torch / C++ types.
 *  - every pointer is a DEVICE pointer unless the name ends in _host.
 *  - the caller owns and allocates every buffer, including workspaces (the *_bytes functions
 *    size them).  The library never allocates, frees or retains a pointer.
 *  - every call is asynchronous on `stream` and never synchronises.
 *  - return value: 0 on success, negative trs_status otherwise; the message of the last failure
 *    on the calling thread is available from trs_last_error().  No exception crosses the ABI.
 *  - ids are int64 ("LongTensor", dataset/dataset.py:268-272), parameters are fp32 row-major
 *    [n_rows, dim] exactly as nn.Embedding stores them; the kernels update them in place.
 */
#ifndef TRS_H_
#define TRS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRS_ABI_VERSION 1
#define TRS_MAX_META 8 /* metadata features (columns) per model */

typedef struct CUstream_st* trs_stream_t; /* == cudaStream_t */

typedef enum {
    TRS_OK = 0,
    TRS_ERR_ARG = -1,     /* bad argument (null pointer, unsupported dim, ...) */
    TRS_ERR_CUDA = -2,    /* a CUDA runtime call failed */
    TRS_ERR_WORKSPACE = -3 /* caller workspace too small */
} trs_status;

typedef enum { TRS_NET_LINEAR = 0, TRS_NET_FM = 1, TRS_NET_MLP = 2 } trs_net;
typedef enum { TRS_OPT_SGD = 0, TRS_OPT_ADAGRAD = 1, TRS_OPT_SPARSE_ADAM = 2 } trs_opt;

/* One id space = an embedding table [n_rows, dim] plus (optionally) the width-1 table that is
 * always looked up with the same ids (Linear: user_bias/item_bias, linear.py:45-51; FM:
 * linear_user/linear_item/linear_metadata, fm.py:42-56).  s0/s1 are the optimizer state tensors
 * of the same shape as their parameter: Adagrad `sum` -> s0; SparseAdam `exp_avg` -> s0,
 * `exp_avg_sq` -> s1; unused ones are NULL. */
typedef struct {
    float* emb;
    float* emb_s0;
    float* emb_s1;
    float* lin; /* [n_rows, 1] or NULL */
    float* lin_s0;
    float* lin_s1;
    int64_t n_rows;
} trs_table;

typedef struct {
    int32_t net;    /* trs_net */
    int32_t dim;    /* n_factors */
    int32_t n_meta; /* F: metadata features, 0..TRS_MAX_META */
    int32_t reserved;
    trs_table user;
    trs_table item;
    trs_table meta[TRS_MAX_META];
} trs_model;

/* The (already shuffled) samples of one epoch, as the reference loader would emit them batch
 * after batch (dataset/dataset.py:414-458): step s covers samples [s*batch, min((s+1)*batch, n)).
 * Metadata ids are one id per feature, row-major [n_samples, n_meta]. */
typedef struct {
    const int64_t* user;
    const int64_t* pos;
    const int64_t* neg;
    const int64_t* pos_meta; /* NULL when n_meta == 0 */
    const int64_t* neg_meta;
    int64_t n_samples;
    int32_t batch;
    int32_t reserved;
} trs_epoch;

/* Row-wise optimizer (torch.optim.{SGD,Adagrad,SparseAdam} on sparse gradients;
 * torch: optim/_functional.py:24-84, optim/adagrad.py:363-373, optim/sgd.py).
 * step_scale[s] is the scalar the update of step s is multiplied by, computed by the host in
 * double exactly as torch does and rounded to fp32: SGD lr; Adagrad clr = lr/(1+(t-1)*lr_decay);
 * SparseAdam lr*sqrt(1-beta2^t)/(1-beta1^t). */
typedef struct {
    int32_t kind; /* trs_opt */
    int32_t reserved;
    double beta1; /* python floats of the torch optimizer; (1-beta) is rounded to fp32 inside */
    double beta2;
    double eps;
    const float* step_scale; /* device, [>= first_step + n_steps] */
} trs_optim;

/* ---- library ------------------------------------------------------------------------- */
int trs_abi_version(void);
const char* trs_last_error(void);
/* SM count and the persistent grid the training kernel would use on the current device. */
int trs_device_info(int* sm_count_host, int* train_grid_host, int* train_block_host);

/* ---- a1: embedding rows (embeddings/init_embeddings.py:5,53 -> aten::embedding) -------- */
/* out[b,:] = table[idx[b],:] (+ sum_f meta_emb[f][meta_idx[b,f],:]) -- 128-bit row gather that
 * sum-pools the metadata rows into the item row (linear.py:67-75).  Bit-exact. */
int trs_embed_gather_sum(const float* table, int dim, const int64_t* idx, int64_t n,
                         const float* const* meta_tables_host, const int64_t* meta_idx, int n_meta,
                         float* out, trs_stream_t stream);

/* ---- a2/a3: scorer forward (linear.py:54-80 -> (B,1); fm.py:60-101 -> (B,)) ------------- */
int trs_scores(const trs_model* model, const int64_t* user, const int64_t* item,
               const int64_t* meta, int64_t n, float* out, trs_stream_t stream);

/* ---- a9: dynamic negatives (dataset/dataset.py:435-447) on device, Philox4x32-10 --------- */
/* neg[j] ~ U[0, n_items) redrawn while == pos[j]; counter = first_index + j, key = seed.
 * If item_meta ([n_items, n_meta]) is given, also emits neg_meta[j,:] = item_meta[neg[j],:]
 * (dataset.py:375-411).  Bit-exact against oracle/cf_oracle.py:philox_negatives. */
int trs_philox_negatives(uint64_t seed, uint64_t first_index, const int64_t* pos, int64_t n,
                         int64_t n_items, const int64_t* item_meta, int n_meta, int64_t* neg,
                         int64_t* neg_meta, trs_stream_t stream);

/* ids in [0, n_rows)?  Adds the number of offenders to *bad_count (device int32). */
int trs_validate_ids(const int64_t* ids, int64_t n, int64_t n_rows, int32_t* bad_count,
                     trs_stream_t stream);

/* ---- a7 (K5): the sort half of coalesce(), for a whole epoch at once ---------------------- */
/* For every step and every id space, a stable sort of that step's lookups by row id (what
 * grad.coalesce() does per step, torch: optim/_functional.py:44).  `plan` receives the sorted
 * (row, lookup) pairs; `tmp` is scratch of trs_plan_tmp_bytes().  One call takes at most 65535 steps
 * (TRS_ERR_ARG beyond): a longer epoch is passed as consecutive runs of whole steps, as the host mirror does. */
size_t trs_plan_bytes(const trs_model* model, const trs_epoch* epoch);
size_t trs_plan_tmp_bytes(const trs_model* model, const trs_epoch* epoch);
int trs_plan_build(const trs_model* model, const trs_epoch* epoch, void* plan, size_t plan_bytes,
                   void* tmp, size_t tmp_bytes, trs_stream_t stream);

/* ---- a6+a5+a7: fused fwd + hinge + bwd + segmented reduce + row-wise optimizer ------------ */
/* Runs steps [first_step, first_step+n_steps) of the epoch in ONE persistent cooperative
 * launch (model.py:274-284 per step: forward x2, hinge_loss, backward, optimizer.step()).
 * loss[s] receives the batch-mean hinge of step first_step+s (the value loss.item() returns at
 * model.py:200), without a host sync. */
size_t trs_train_workspace_bytes(const trs_model* model, const trs_epoch* epoch);
int trs_train_steps(const trs_model* model, const trs_epoch* epoch, const trs_optim* optim,
                    const void* plan, void* workspace, size_t workspace_bytes, int first_step,
                    int n_steps, float* loss, trs_stream_t stream);

/* ---- a10: evaluate (model.py:292-338, evaluate/metrics.py:23-31) -------------------------- */
/* Per batch b of `epoch`: loss[b] = mean hinge, auc[b] = #(pos > neg)/len.  pos_out/neg_out
 * (nullable) receive the raw scores. */
int trs_eval_pairwise(const trs_model* model, const trs_epoch* epoch, float* loss, float* auc,
                      float* pos_out, float* neg_out, trs_stream_t stream);

/* ---- a4 (K7): dense layers of the MLP tower (collaborative/mlp.py:74-85, 107-113) ------------ */
/* out[m, n] = sum_k a[m, k] * b[n, k] (+ bias[n]) on the tcgen05 tensor cores: bf16 operands, both
 * contiguous along k, fp32 accumulation in TMEM.  nn.Linear forward is (a = activations, b = weight);
 * dgrad and wgrad reach the same form through transposed operand copies (see DESIGN.md).
 *  - out is fp32 or bf16 (out_bf16), row-major with leading dimension ldc.
 *  - splits > 1 cuts k into `splits` ranges; split z writes its raw fp32 partial at out + z*split_stride.
 *  - col_sum / col_sumsq (nullable, [ceil(m/128), n]): per 128-row tile, the column sums of the stored
 *    output and of its squares over the valid rows, for BatchNorm1d batch statistics (mlp.py:82, 109).
 *    A row is valid iff (row % rows_per_half) < rows_valid (the positive and the negative pass of a
 *    step are stacked, each padded to rows_per_half rows); rows_per_half == 0: every row is valid.
 *  - a_mn / b_mn: the operand is given transposed in memory ([k, m] / [k, n]); the tensor cores read it
 *    "MN-major", so dgrad (b = W as stored) and wgrad (a = dZ, b = activations, both as stored) need no
 *    transposed copies.  Supported: (0,0), (0,1), (1,1); a_mn writes fp32 only.
 *  k, n and ldc must be multiples of 8; a and b 16-byte aligned. */
typedef struct {
    const void* a; /* bf16 [m, k], leading dimension lda */
    const void* b; /* bf16 [n, k], leading dimension ldb */
    int64_t lda, ldb;
    int64_t m, n, k;
    void* out;
    int64_t ldc;
    int64_t split_stride;
    int32_t out_bf16;
    int32_t splits;
    int32_t a_mn; /* a is stored [k, m] (m contiguous, leading dimension lda) instead of [m, k] */
    int32_t b_mn; /* b is stored [k, n] */
    const float* bias;
    float* col_sum;
    float* col_sumsq;
    int64_t rows_per_half;
    int64_t rows_valid;
} trs_gemm_args;
int trs_gemm_bf16_tn(const trs_gemm_args* args, trs_stream_t stream);

/* ---- a4 + a6 + a7 for net_type='mlp' (collaborative/mlp.py:88-115, model.py:171-200) --------- */
/* The tower: concat[user, item, metadata_f...] -> (Linear -> BatchNorm1d -> ReLU) x n_layers ->
 * Linear(-> 1).  Pointers are the fp32 parameters / buffers of the torch modules (fcs.l, bns.l,
 * output_layer; collaborative/mlp.py:74-85), d* receive the dense gradients of one training step, and
 * s0* are the dense optimizer state (Adagrad `sum`; NULL for SGD) updated in place together with the
 * parameters.  The embedding tables travel in a trs_model with net = TRS_NET_MLP (lin pointers NULL). */
#define TRS_MAX_LAYERS 8
typedef struct {
    int32_t n_layers; /* hidden layers, 1..TRS_MAX_LAYERS */
    int32_t use_bn;
    int32_t hidden[TRS_MAX_LAYERS];
    float* W[TRS_MAX_LAYERS];     /* [hidden[l], in_l], in_0 = dim*(2+n_meta), in_l = hidden[l-1] */
    float* b[TRS_MAX_LAYERS];     /* [hidden[l]] */
    float* gamma[TRS_MAX_LAYERS]; /* BatchNorm1d weight / bias / running stats (use_bn) */
    float* beta[TRS_MAX_LAYERS];
    float* running_mean[TRS_MAX_LAYERS];
    float* running_var[TRS_MAX_LAYERS];
    float* w_out; /* [1, hidden[n_layers-1]] */
    float* b_out; /* [1] */
    /* training only */
    float* dW[TRS_MAX_LAYERS];
    float* db[TRS_MAX_LAYERS];
    float* dgamma[TRS_MAX_LAYERS];
    float* dbeta[TRS_MAX_LAYERS];
    float* dw_out;
    float* db_out;
    float* s0W[TRS_MAX_LAYERS];
    float* s0b[TRS_MAX_LAYERS];
    float* s0gamma[TRS_MAX_LAYERS];
    float* s0beta[TRS_MAX_LAYERS];
    float* s0w_out;
    float* s0b_out;
} trs_mlp;

/* Forward of n (user, item[, meta]) rows -> out[n] (net.forward, mlp.py:88-115).  batch_stats = 0: eval
 * mode (BatchNorm uses running statistics); 1: train mode (this call's batch statistics, running
 * statistics updated once, as one reference forward pass does). */
size_t trs_mlp_forward_workspace_bytes(const trs_model* model, const trs_mlp* mlp, int64_t n);
int trs_mlp_forward(const trs_model* model, const trs_mlp* mlp, const int64_t* user, const int64_t* item,
                    const int64_t* meta, int64_t n, int batch_stats, float* out, void* workspace,
                    size_t workspace_bytes, trs_stream_t stream);

/* Steps [first_step, first_step+n_steps) of the epoch (model.py:274-284): both passes forward with
 * per-pass BatchNorm statistics (running statistics updated twice per step), hinge, backward through the
 * tcgen05 GEMMs, dense update (SGD / Adagrad) of the tower, deterministic segmented reduce + row-wise
 * update of the embedding tables.  No host synchronisation; loss[s] as in trs_train_steps.
 * `plan` comes from trs_plan_build on the same model / epoch. */
size_t trs_mlp_train_workspace_bytes(const trs_model* model, const trs_mlp* mlp, const trs_epoch* epoch);
int trs_mlp_train_steps(const trs_model* model, const trs_mlp* mlp, const trs_epoch* epoch,
                        const trs_optim* optim, const void* plan, void* workspace, size_t workspace_bytes,
                        int first_step, int n_steps, float* loss, trs_stream_t stream);

/* ---- a11: predict (model.py:341-452) batched over users: top-k items per user against ALL items ------ */
/* For each query user users[q]: out_idx[q, 0..k) = item ids (+ item_offset) of the k best scores, best
 * first, ties broken towards the lower item id (== torch.sort(stable=True, descending=True) on the
 * scores trs_scores returns); out_score[q, :] those fp32 scores.  Phase 1 scores user tiles against every
 * item on the tcgen05 tensor cores (bf16) with the top-k filter fused into the epilogue and keeps a
 * provable superset of the exact top-k; phase 2 re-scores the survivors in fp32 (csrc/topk.cu).
 * overflow[q] != 0 marks a user whose candidate superset did not fit (e.g. thousands of tied, saturated
 * FM scores): its output row is invalid and the caller must rank that user with trs_scores + sort.
 * item_meta ([n_items, n_meta], NULL without metadata) gives every item's metadata ids.
 * Linear and FM only (the MLP tower does not factorise into user x item). 1 <= k <= 128. */
size_t trs_predict_topk_workspace_bytes(const trs_model* model, int64_t n_query, int k);
int trs_predict_topk(const trs_model* model, const int64_t* users, int64_t n_query, const int64_t* item_meta,
                     int k, int64_t item_offset, int64_t* out_idx, float* out_score, int32_t* overflow,
                     void* workspace, size_t workspace_bytes, trs_stream_t stream);
/* The same with the caller's promise `items_prepared` != 0: `workspace` was last used by a call with the same item
 * tables (contents unchanged), item_meta and n_query, so the prepared bf16 item operand inside it is still valid and
 * is not rebuilt -- serving many user batches against an unchanged model (model.py:383 loops the same way). */
int trs_predict_topk_reuse(const trs_model* model, const int64_t* users, int64_t n_query, const int64_t* item_meta,
                           int k, int64_t item_offset, int64_t* out_idx, float* out_score, int32_t* overflow,
                           void* workspace, size_t workspace_bytes, int items_prepared, trs_stream_t stream);

/* ---- multi-GPU building blocks (SURVEY.md §8e; the reference is single-device, model.py:74) ----------- */
/* a7 for the OWNER of a table shard: grad.coalesce() + the row-wise optimizer step (torch:
 * optim/_functional.py:44-84, optim/adagrad.py:363-373) on an explicit list of n (row id, gradient row)
 * pairs, e.g. the gradient rows other ranks sent.  Duplicate rows are summed in list order after a stable
 * sort by id (deterministic); grad_lin (nullable) is the gradient of the width-1 companion table.
 * optim->step_scale[step] scales the update as in trs_train_steps. */
size_t trs_sparse_update_workspace_bytes(int64_t n);
int trs_sparse_row_update(const trs_table* table, int dim, const int64_t* ids, int64_t n, const float* grad_rows,
                          const float* grad_lin, const trs_optim* optim, int step, void* workspace,
                          size_t workspace_bytes, trs_stream_t stream);

/* Linear scorer forward x2 + hinge + backward (linear.py:54-80, loss.py:5-9) on rows gathered elsewhere:
 * u/pos/neg rows [batch, dim] and their biases [batch] in, one gradient row per lookup out
 * (g = [hinge >= 0] * inv_batch; d user_bias = 0, SURVEY D12); *loss_sum = sum of the batch's hinges.
 * workspace: at least 8 * SM-count floats. */
int trs_linear_rows_step(int dim, int64_t batch, float inv_batch, const float* u_rows, const float* pos_rows,
                         const float* neg_rows, const float* u_bias, const float* pos_bias, const float* neg_bias,
                         float* g_u, float* g_pos, float* g_neg, float* g_pos_bias, float* g_neg_bias,
                         float* loss_sum, float* workspace, size_t workspace_floats, trs_stream_t stream);

/* Merge n_lists per-shard top-k lists (score / idx laid out [n_lists, n_query, k], idx < 0 = padding) into
 * the global top-k per user, ordered by (score descending, item id ascending) -- the allgather half of the
 * item-sharded predict. n_lists * k <= 4000. */
int trs_topk_merge(const float* score, const int64_t* idx, int n_lists, int k, int64_t n_query,
                   int64_t* out_idx, float* out_score, trs_stream_t stream);

/* ---- a7 for callers that drive autograd themselves: TorchRecSys.forward -> hinge_loss -> backward (model.py:171-200) */
/* Backward of trs_scores (Linear / FM): grad_out[b] = d loss / d score[b]; writes ONE gradient row per lookup --
 * g_user / g_item [n, dim], g_meta[f] [n, dim], and (nullable) the width-1 companions' gradients g_lin_* [n] -- exactly
 * the (index, value) pairs the reference's nn.Embedding(sparse=True) backward emits (uncoalesced; torch's optimizers
 * coalesce).  The host wraps them as sparse COO tensors so that ANY torch optimizer can step on them. */
int trs_scores_backward(const trs_model* model, const int64_t* user, const int64_t* item, const int64_t* meta, int64_t n,
                        const float* grad_out, float* g_user, float* g_item, float* const* g_meta_host,
                        float* g_lin_user, float* g_lin_item, float* const* g_lin_meta_host, trs_stream_t stream);

/* ---- a10 (north_star): sort-based ROC-AUC on the device --------------------------------------------------- */
/* auc_out[0] (device double) = P(score+ > score-) + 0.5 P(score+ == score-) over all n_pos x n_neg pairs, computed as
 * the Mann-Whitney U statistic: radix sort of the n_pos + n_neg scores, tie-averaged ranks, exact integer rank sum
 * (equals sklearn.metrics.roc_auc_score, which the reference's legacy helper/evaluate.py:8-18 calls).  NaN for an
 * empty class.  n_pos + n_neg <= 2^23 per call.  workspace: trs_sort_workspace_bytes(n_pos + n_neg). */
size_t trs_sort_workspace_bytes(int64_t n);
int trs_sorted_auc(const float* pos, int64_t n_pos, const float* neg, int64_t n_neg, double* auc_out, void* workspace,
                   size_t workspace_bytes, trs_stream_t stream);

/* ---- a9: the loader's per-epoch shuffle (dataset/dataset.py:359-373, 420-427) ------------------------------ */
/* perm = a pseudo-random permutation of [0, n): Philox4x32-10 keys (key = seed, counter = position), stable radix
 * sort.  n <= 2^23 per call; workspace: trs_sort_workspace_bytes(n). */
int trs_epoch_shuffle(uint64_t seed, int64_t n, int64_t* perm, void* workspace, size_t workspace_bytes,
                      trs_stream_t stream);
/* dst[c][k, :] = src[c][perm[k], :] for up to 8 int64 id columns of `width[c]` ids per sample at once (what
 * FastDataLoader.__next__ does per key and batch with tensor[current_indices]). */
int trs_gather_rows_i64(const int64_t* const* src_host, int64_t* const* dst_host, const int32_t* width_host, int n_cols,
                        const int64_t* perm, int64_t n, trs_stream_t stream);

/* ---- e1: row-sharded training over PEER-MAPPED table shards (SURVEY.md §8e, BASELINE configs[3]) ------------ */
/* The reference is single-device (model.py:74); this is the multi-GPU form of model.py:274-284 for
 * net_type='linear'.  Row r of the user / item table lives on rank r % world at local row r / world.  Every rank
 * maps every other rank's shard, gradient staging buffer and barrier words into its own address space (CUDA IPC,
 * trs_ipc_* below) and ONE persistent kernel per rank runs K steps:
 *   phase A  the rank's samples of the step (those whose USER row it owns: user rows never cross NVLink): item
 *            rows are read straight from their owner's HBM over NVLink (cp.async from the peer pointer), both
 *            scores, hinge over the GLOBAL batch, and each lookup's gradient row is stored straight into its
 *            owner's staging buffer at slot = the lookup's index in the global batch
 *   cross-rank barrier (flag words in peer memory)
 *   phase B  every owner reduces the staged rows of each of ITS touched rows in slot order (what coalesce() gives;
 *            deterministic) and applies SGD / Adagrad / SparseAdam to its shard
 *   cross-rank barrier
 * No NCCL call on the step path: the exchange IS the kernel's loads and stores. */
#define TRS_MAX_RANKS 8
#define TRS_SHARD_SYNC_BYTES 4096 /* barrier words of one rank; zeroed ONCE when allocated, never afterwards */

typedef struct {
    int32_t rank, world;
    int32_t dim, reserved;
    int64_t n_users, n_items;      /* GLOBAL row counts */
    trs_table user[TRS_MAX_RANKS]; /* rank q's shard as mapped into THIS process (q == rank: plain device memory); */
    trs_table item[TRS_MAX_RANKS]; /*   n_rows = rows of that shard; lin = user_bias / item_bias                  */
    void* stage[TRS_MAX_RANKS];    /* rank q's gradient staging buffer, trs_shard_stage_bytes() */
    void* sync[TRS_MAX_RANKS];     /* rank q's barrier words, TRS_SHARD_SYNC_BYTES */
} trs_shard;

/* `epoch` below is always the GLOBAL epoch: the ids of every rank's samples in loader order, identical on all
 * ranks (an all-gather of the loader output, once per epoch); epoch->batch is the GLOBAL batch.  Metadata is not
 * supported on this path. */
/* Two copies of [global_batch, dim] + [2 * global_batch, dim] + [2 * global_batch] floats: even and odd steps use
 * different copies, so a rank may store step s+1's gradient rows into a peer that is still reading step s's. */
size_t trs_shard_stage_bytes(int dim, int global_batch);
/* The rank's plan: which samples it runs (user % world == rank) with their flags (user row looked up once in the
 * step; user / positive / negative row updated by the step before), and, per step, the (local row, slot) pairs of
 * the lookups it OWNS and still has to apply after the samples ran, stably sorted by row. */
size_t trs_shard_plan_bytes(const trs_epoch* epoch);
size_t trs_shard_plan_tmp_bytes(const trs_epoch* epoch);
int trs_shard_plan_build(const trs_shard* shard, const trs_epoch* epoch, void* plan, size_t plan_bytes, void* tmp,
                         size_t tmp_bytes, trs_stream_t stream);
/* Steps [first_step, first_step + n_steps) for the n_local ranks this launch hosts: 1 in production (one process
 * per GPU); all `world` ranks when a single GPU emulates the group (tests: one cooperative launch, the SMs split
 * between the ranks -- separate launches must never wait on each other on one device).
 *  - sync_epoch: cross-rank barriers the group has passed so far (2 per step); the caller adds 2 * n_steps after
 *    every call, identically on every rank.
 *  - loss_sum[i][s]: sum of the hinges of rank i's samples of step first_step + s (all-reduce and divide by the
 *    step's global sample count for the value loss.item() returns at model.py:200).
 *  - status (device int32, zeroed by the caller): set non-zero if a peer did not arrive within timeout_ms (the
 *    kernel then stops waiting and finishes; the tables are garbage and the caller must raise). */
size_t trs_shard_workspace_bytes(const trs_epoch* epoch, int n_local);
int trs_shard_train_steps(const trs_shard* shards, int n_local, const trs_epoch* epoch, const trs_optim* optim,
                          const void* const* plans_host, void* workspace, size_t workspace_bytes, int first_step,
                          int n_steps, uint64_t sync_epoch, float* const* loss_sum_host, int32_t* status,
                          int timeout_ms, trs_stream_t stream);

/* Serving on the shards where they live: every row is read from its owner through the pointers of `shard` (peer
 * mappings), nothing is gathered.  Ids must lie in [0, n_users) / [0, n_items).  The caller orders these reads
 * against the owners' next training launch (sharded.py ends each serving call with a group collective). */
/* a10 (model.py:292-338) for batches [first_batch, first_batch + n_batches) of the global epoch: loss[b - first_batch]
 * and auc[b - first_batch] as trs_eval_pairwise computes them on the gathered model, bit for bit; pos_out / neg_out
 * (nullable) receive the raw scores from the range's first sample on. */
int trs_shard_eval_pairwise(const trs_shard* shard, const trs_epoch* epoch, int64_t first_batch, int64_t n_batches,
                            float* loss, float* auc, float* pos_out, float* neg_out, trs_stream_t stream);
/* emb_out[j, :] = row ids[j] of the user (table 0) or item (table 1) table, lin_out[j] (nullable) = its bias, both
 * copied bit for bit from the owner. */
int trs_shard_gather_rows(const trs_shard* shard, int table, const int64_t* ids, int64_t n, float* emb_out,
                          float* lin_out, trs_stream_t stream);
/* Exact top-k of rank shard->rank's OWN item shard for n_query dense query rows user_emb [n_query, dim] / user_lin
 * [n_query] (nullable; e.g. from trs_shard_gather_rows): out_idx[q, 0..k) = GLOBAL item ids (local * world + rank) of
 * the k best scores, out_score[q, :] those fp32 scores, equal bit for bit to trs_scores on the gathered model, ordered
 * by (score desc, id asc) with equal values as ties (torch.sort(stable=True, descending=True)); slots with no item are
 * -1 / -inf.  1 <= k <= 1024.  excl_ptr [n_query + 1] / excl_ids (both nullable): per query position, the sorted LOCAL
 * item ids of this shard to leave out.  Reads only the rank's own shard.  workspace: the _workspace_bytes size (0 =
 * bad arguments, see trs_last_error). */
size_t trs_shard_topk_exact_workspace_bytes(const trs_shard* shard, int64_t n_query, int k);
int trs_shard_topk_exact(const trs_shard* shard, const float* user_emb, const float* user_lin, int64_t n_query, int k,
                         const int64_t* excl_ptr, const int64_t* excl_ids, int64_t* out_idx, float* out_score,
                         void* workspace, size_t workspace_bytes, trs_stream_t stream);
/* Merge n_lists sorted lists (score / idx [n_lists, n_query, k_in], each row ordered by (score desc, id asc), idx < 0 =
 * padding at the end) into out [n_query, k_out] in the same order, -1 / -inf padded.  excl_ptr [n_query + 1] /
 * excl_ids (both nullable): per query, sorted ids (in the lists' id space) to drop.  O(n_lists^2 k_in log k_in) per
 * query; n_lists * (k_in + 1) <= 40960. */
int trs_shard_topk_merge_sorted(const float* score, const int64_t* idx, int n_lists, int64_t n_query, int k_in,
                                int k_out, const int64_t* excl_ptr, const int64_t* excl_ids, int64_t* out_idx,
                                float* out_score, trs_stream_t stream);

/* CUDA IPC plumbing for the peer mapping (the only entry points that touch address spaces; they never allocate
 * device memory).  export: 64-byte handle of the allocation that contains `ptr` + the offset of ptr inside it;
 * open: maps that allocation into this process (peer access enabled lazily) and returns its base; close unmaps. */
int trs_ipc_export(const void* ptr, void* handle64_host, uint64_t* offset_host);
int trs_ipc_open(const void* handle64_host, void** base_host);
int trs_ipc_close(void* base);

#ifdef __cplusplus
}
#endif
#endif /* TRS_H_ */
