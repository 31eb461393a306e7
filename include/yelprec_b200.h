/*
 * yelprec_b200.h — C ABI of the B200-native BPR-MF / NGCF train + full-catalog eval hot path.
 *
 * One shared library (libyelprec_b200.so), extern "C", plain pointers and sizes only.
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _h;
 *   - every call enqueues work on `stream` (a cudaStream_t passed as void*) and returns without
 *     synchronising; nothing is allocated inside the library: callers own all buffers;
 *   - return value: 0 = ok, 1..999 = cudaError_t of the launch, >=1000 = yr_status (bad argument);
 *   - embedding tables are fp32 row-major [rows x d]; ids are int64 exactly as the reference's
 *     default-collated batches (data/datasets/mf_dataset.py:26-31);
 *   - "reference" citations are relative to twndus/YelpRecommendation.
 *
 * The reference has no FFI of its own (pure Python/PyTorch); each entry point below names the
 * reference interface whose body it replaces. INTEGRATION.md shows the ctypes stub a maintainer adds.
 */
#ifndef YELPREC_B200_H
#define YELPREC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* yr_stream; /* cudaStream_t */

enum yr_status {
  YR_OK = 0,
  YR_ERR_BAD_ARG = 1000,      /* null pointer / non-positive size */
  YR_ERR_BAD_DIM = 1001,      /* embedding width not supported by the kernels */
  YR_ERR_BAD_OPT = 1002,      /* unknown optimizer kind (reference: NotImplementedError, base_trainer.py:41-43) */
  YR_ERR_WORKSPACE = 1003,    /* workspace too small */
  YR_ERR_COOP = 1004          /* device cannot co-schedule the cooperative grid */
};

enum yr_opt_kind { YR_OPT_SGD = 0, YR_OPT_ADAM = 1, YR_OPT_ADAMW = 2 };

/* Optimizer hyper-parameters with torch.optim defaults semantics (trainers/base_trainer.py:34-40).
 * `step` is the 1-based index of the FIRST optimizer step the call performs (Adam bias correction). */
typedef struct yr_opt {
  int32_t kind;
  int32_t step;
  double lr, weight_decay, beta1, beta2, eps;
} yr_opt;

/* Library / device info. */
int yr_version(void);
int yr_device_sm_count(int* sm_count_h);

/* ------------------------------------------------------------------------------------------------
 * BPR-MF  (models/mf.py, loss.py, trainers/mf_trainer.py)
 * ---------------------------------------------------------------------------------------------- */

/* MatrixFactorization.forward (models/mf.py:20-23): out[b] = sum_k U[uid[b],k] * V[iid[b],k],
 * accumulated as one fp32 fma chain k = 0..d-1 (the canonical order the oracle uses).
 * Out-of-range ids set *err (sticky, non-zero) instead of reading out of bounds. */
int yr_mf_score(const float* U, const float* V, int64_t nU, int64_t nI, int d,
                const int64_t* uid, const int64_t* iid, int64_t B, float* out, int32_t* err,
                yr_stream stream);

/* Backward of yr_mf_score for autograd users (an unmodified reference trainer calling
 * loss.backward(), trainers/mf_trainer.py:111): gU[uid[b]] += gout[b]*V[iid[b]], gV[iid[b]] += gout[b]*U[uid[b]].
 * gU/gV are dense [rows x d] and are accumulated into (caller zeroes them). */
int yr_mf_score_bwd(const float* U, const float* V, int64_t nU, int64_t nI, int d,
                    const int64_t* uid, const int64_t* iid, int64_t B, const float* gout,
                    float* gU, float* gV, yr_stream stream);

/* BPRLoss.forward (loss.py:25-27): *loss = mean_b( -logsigmoid(pos[b]-neg[b]) ). */
int yr_bpr_loss_fwd(const float* pos, const float* neg, int64_t B, float* loss, yr_stream stream);
/* d loss / d pos, d loss / d neg scaled by *gloss (device scalar). */
int yr_bpr_loss_bwd(const float* pos, const float* neg, int64_t B, const float* gloss,
                    float* gpos, float* gneg, yr_stream stream);

/* State of the fused trainer: parameters, optimizer moments and scratch.
 * flagU / flagV must be all-zero on first use; every call leaves them all-zero again. */
typedef struct yr_mf_state {
  float *U, *V;             /* [nU x d], [nI x d] */
  float *mU, *vU, *mV, *vV; /* Adam exp_avg / exp_avg_sq, same shapes (unused for SGD, may be NULL) */
  int32_t *flagU, *flagV;   /* [nU], [nI]: row -> position of its segment in the step's sorted id lists (dense-semantics steps) */
  int32_t *counters;        /* 64-byte block, zero on first use (parity of the next step) */
  int32_t *err;             /* [1] sticky bad-id flag (reference: IndexError from nn.Embedding) */
  void *ws; size_t ws_bytes;/* >= yr_bpr_mf_train_ws_bytes(n_triples, B, d) of the call: sorted id lists of every batch,
                               per-triple gradient rows of one step, per-CTA loss partials */
  int64_t nU, nI;
  int32_t d;
  int32_t deterministic;    /* != 0: plain-SGD steps also take the ordered (atomics-free) path, see below */
} yr_mf_state;

/* MFTrainer.train hot loop (trainers/mf_trainer.py:100-116) for `n_triples` pre-collated triples cut
 * into consecutive batches of B (last one short, as DataLoader keeps it, train.py:76): per batch
 * forward x2, BPR loss, gradient with duplicate rows summed, ONE optimizer update per row
 * (SGD / Adam / AdamW with torch dense semantics), all inside one persistent cooperative kernel.
 * Summation order of duplicate rows = the reference's on the CPU: per embedding call sequentially in batch order
 * (embedding_dense_backward), then the two calls added (AccumulateGrad); the loss is a fixed-order double sum.
 * Results are bit-identical from run to run and to oracle/yr_oracle.c — except plain SGD (wd = 0) with
 * B <= resident warps and deterministic == 0, which keeps gradients in registers and applies them as vector REDs
 * (duplicates summed in arrival order, ulp-level differences).
 * loss_sum (double, device) += sum over batches of the batch-mean loss (quirk Q1);
 * step_loss (float, device, may be NULL) receives every batch mean. */
size_t yr_bpr_mf_train_ws_bytes(int64_t n_triples, int32_t B, int d);
int yr_bpr_mf_train(const yr_mf_state* st, const yr_opt* opt,
                    const int64_t* uid, const int64_t* pos, const int64_t* neg,
                    int64_t n_triples, int32_t B, double* loss_sum, float* step_loss,
                    yr_stream stream);

/* MFTrainer.validate (trainers/mf_trainer.py:118-132): same batching, forward + loss only. */
int yr_bpr_mf_validate(const float* U, const float* V, int64_t nU, int64_t nI, int d,
                       const int64_t* uid, const int64_t* pos, const int64_t* neg,
                       int64_t n_triples, int32_t B, double* loss_sum, float* step_loss,
                       int32_t* err, yr_stream stream);

/* ------------------------------------------------------------------------------------------------
 * NGCF  (models/ngcf.py, trainers/ngcf_trainer.py)
 * ---------------------------------------------------------------------------------------------- */

/* CSR matrix (int32 indices, fp32 values) plus its load-balancing plan. Rows longer than YR_SPMM_CHUNK
 * non-zeros are cut into chunks of YR_SPMM_CHUNK consecutive non-zeros so that one warp never walks more than
 * that (the Yelp-shape graph has item rows with > 10,000 non-zeros). The plan is built once per graph on the
 * host (yr_spmm_plan_*_h) and uploaded by the caller.
 * Canonical summation order (the oracle restates it): a row with <= YR_SPMM_CHUNK non-zeros is ONE fma chain in
 * CSR order (starting from Y's old value when accumulating); a longer row is the left-to-right sum of its chunk
 * partials, each chunk one fma chain from 0 (and Y_old + that sum when accumulating). */
#define YR_SPMM_CHUNK 128
typedef struct yr_csr {
  int64_t n_rows, nnz;
  const int32_t *rowptr, *col;
  const float* val;
  int32_t n_chunks;               /* work items: one per short row, ceil(len/CHUNK) per long row */
  const int32_t *chunk_desc;      /* [n_chunks x 4], 16-byte aligned: {row, first non-zero, length | split_row_index << 8
                                     (| 1 << 31 for a big row), slot} — slot -1 = whole row (direct store), else index into
                                     `partials` */
  int32_t n_split_rows;           /* rows that were cut */
  const int32_t *split_row;       /* [n_split_rows] */
  const int32_t *split_ptr;       /* [n_split_rows+1] range of partial slots of each split row */
  float* partials;                /* [split_ptr[n_split_rows] x d] scratch */
  int32_t* split_count;           /* [n_split_rows] arrival counters, zero on first use; every call leaves them zero.
                                     The chunk that arrives last at a split row sums that row's partials (in order). */
  int32_t n_big_rows;             /* split rows with more than YR_SPMM_BIG_CHUNKS chunks (hub rows of a scaled graph): their */
  const int32_t* big_split_idx;   /* partials are summed — same left-to-right order — by a follow-up kernel that stages them
                                     through shared memory instead of one warp walking thousands of partials; [n_big_rows]
                                     indices into split_row / split_ptr, from yr_spmm_plan_big_h. 0 / NULL if there are none. */
  int32_t reserve_sms;            /* 0: the SpMM fills the GPU. R > 0: it runs as (SM count - R) persistent 1,024-thread CTAs,
                                     one per SM, and leaves R SMs empty — for the NCCL kernels of a panel exchange that is meant
                                     to run underneath it (kernels that need an empty SM never start behind a grid of small
                                     CTAs that keeps refilling every SM). Same arithmetic, same results. */
} yr_csr;

/* Host-side plan builder (host pointers). Call _size_h first, allocate, then _fill_h. */
int yr_spmm_plan_size_h(const int32_t* rowptr_h, int64_t n_rows, int32_t* n_chunks_h, int32_t* n_split_rows_h,
                        int32_t* n_partials_h);
int yr_spmm_plan_fill_h(const int32_t* rowptr_h, int64_t n_rows, int32_t* chunk_desc_h, int32_t* split_row_h,
                        int32_t* split_ptr_h);
/* Split rows with more than YR_SPMM_BIG_CHUNKS chunks: *n_big_h = how many; big_split_idx_h (may be NULL to only count)
 * receives their indices into the split-row list. Their chunk descriptors carry bit 31 of word 2 (set by _fill_h). */
#define YR_SPMM_BIG_CHUNKS 256
int yr_spmm_plan_big_h(const int32_t* rowptr_h, int64_t n_rows, int32_t* n_big_h, int32_t* big_split_idx_h);

/* Y = A X (accumulate == 0) or Y += A X (accumulate != 0), X/Y row-major [n_rows x d].
 * Replaces torch.sparse.mm(laplacian_matrix, last_embed) (models/ngcf.py:64,67). */
int yr_spmm_csr(const yr_csr* A, int d, const float* X, float* Y, int accumulate, yr_stream stream);

/* Where the per-layer d x d transforms run (`dense_mode` argument / yr_ngcf_state.dense_mode — per call and per
 * trainer state, nothing process-wide): YR_DENSE_TC (default of the Python trainers) = forward and backward on tensor
 * cores, tcgen05.mma.kind::tf32 with the 3xTF32 split (within the 1e-5 parity bar; csrc/ngcf_tc.cu, csrc/ngcf_tc_bwd.cu);
 * YR_DENSE_TC_FWD = forward on tensor cores, backward on the FP32 pipe;
 * YR_DENSE_FP32 = FP32 pipe for both, one fma chain per output (forward bit-comparable with the oracle).
 * The tensor-core kernels take d = 64 and d = 128; the transforms accept d in {32, 64, 128} (YR_ERR_BAD_DIM otherwise)
 * and run on the FP32 pipe at d = 32 in every mode. */
enum yr_dense_mode { YR_DENSE_FP32 = 0, YR_DENSE_TC_FWD = 1, YR_DENSE_TC = 2 };
/* Bits 8..15 of a `dense_mode` argument: SMs the tensor-core kernels of that call leave empty (see yr_csr.reserve_sms);
 * 0 = none. YR_DENSE_RESERVE(mode, r) builds the argument. */
#define YR_DENSE_RESERVE(mode, r) ((mode) | (((r) & 0xff) << 8))

/* NGCF.embedding_propagation (models/ngcf.py:60-72) for one layer on the whole graph:
 *   LE = L E;  E_next = leaky_relu( (LE+E) W1^T + (E * LE) W2^T , slope )
 * W1, W2 are nn.Linear weights [d x d] (out x in). LE_save [n x d] receives L E (kept for backward). */
int yr_ngcf_layer_fwd(const yr_csr* L, int d, const float* E, const float* W1, const float* W2, float slope,
                      float* E_next, float* LE_save, int dense_mode, yr_stream stream);

/* Backward of one layer. G_next = dLoss/dE_next. LT is the CSR of L^T.
 *   dZ = G_next * leaky'(E_next); dS = dZ W1; dP = dZ W2;
 *   G += dS + dP*LE + L^T (dS + dP*E);   dW1 = dZ^T (LE+E);  dW2 = dZ^T (E*LE)
 * T [n x d] is scratch for the transposed SpMM operand; ws holds per-CTA dW partials
 * (yr_ngcf_layer_bwd_ws_bytes). dW1/dW2 are OVERWRITTEN with this layer's weight gradient. */
size_t yr_ngcf_layer_bwd_ws_bytes(int d);
int yr_ngcf_layer_bwd(const yr_csr* LT, int d, const float* E, const float* LE, const float* E_next,
                      const float* G_next, const float* W1, const float* W2, float slope,
                      float* G, float* T, float* dW1, float* dW2, void* ws, size_t ws_bytes,
                      int dense_mode, yr_stream stream);

/* The dense halves of the two calls above on n rows, WITHOUT the SpMM (models/ngcf.py:65-72 and its autograd):
 * the row-sharded trainer (BASELINE config 5) runs the SpMM on its row block of L against the all-gathered operand
 * and these on its local rows. yr_ngcf_dense_bwd: G += dS + dP*LE, T = dS + dP*E, dW1/dW2 overwritten. */
int yr_ngcf_dense_fwd(int d, int64_t n, const float* E, const float* LE, const float* W1, const float* W2,
                      float slope, float* E_next, int dense_mode, yr_stream stream);
int yr_ngcf_dense_bwd(int d, int64_t n, const float* E, const float* LE, const float* E_next,
                      const float* G_next, const float* W1, const float* W2, float slope,
                      float* G, float* T, float* dW1, float* dW2, void* ws, size_t ws_bytes,
                      int dense_mode, yr_stream stream);

/* Tail of NGCF.bpr_forward + BPRLoss (models/ngcf.py:37-45, loss.py:25-27) and its backward:
 * rows u / nU+pos / nU+neg are gathered from every layer output E_l (l = 0..n_layers), the concatenated
 * dots give pos/neg scores, the batch-mean loss is added to
 * *loss_sum and written to *step_loss, and, if G_layers != NULL, the row gradients are scatter-added
 * into G_l. E_layers / G_layers are DEVICE arrays of n_layers+1 device pointers. */
/* loss_sum is a device double[2]: [0] += batch mean, [1] is a zeroed scratch accumulator. */
int yr_ngcf_tail(const float* const* E_layers, float* const* G_layers, int n_layers, int64_t nU,
                 int64_t nI, int d, const int64_t* uid, const int64_t* pos, const int64_t* neg,
                 int64_t B, float* pos_out, float* neg_out, double* loss_sum, float* step_loss,
                 int32_t* err, yr_stream stream);

/* One dense torch.optim step over a flat parameter (Adam / AdamW / SGD, single-tensor op order of
 * torch.optim, trainers/base_trainer.py:34-40). m, v may be NULL for SGD. Any n and any 4-byte-aligned pointers
 * (a view that starts inside a tensor); with 16-byte-aligned pointers the step runs on float4 accesses, same bits. */
int yr_dense_opt_step(float* p, const float* g, float* m, float* v, int64_t n, const yr_opt* opt,
                      yr_stream stream);

/* The same step over up to YR_OPT_MAX_TENSORS parameter tensors in ONE launch (host arrays of device pointers and
 * element counts; every count a multiple of 4, every pointer 16-byte aligned). zero_grad != 0 clears each gradient
 * after it has been consumed (optimizer.zero_grad() of the next step, trainers/cdae_trainer.py:42). */
#define YR_OPT_MAX_TENSORS 8
int yr_dense_opt_step_multi(int count, float* const* p, float* const* g, float* const* m, float* const* v,
                            const int64_t* n, const yr_opt* opt, int zero_grad, yr_stream stream);

/* Whole NGCFTrainer.train step (trainers/ngcf_trainer.py:106-115) as one host call: n_layers x layer_fwd,
 * tail (+loss), n_layers x layer_bwd, dense optimizer step over embedding.weight and every W1/W2.
 * All buffers are caller-owned; E[0] is the embedding parameter, E[1..n_layers] the layer outputs. */
#define YR_NGCF_MAX_LAYERS 7
typedef struct yr_ngcf_state {
  int64_t nU, nI;
  int32_t d, n_layers;
  yr_csr L, LT;                       /* CSR (+plan) of L and of L^T */
  float* E[YR_NGCF_MAX_LAYERS + 1];   /* [n x d] each, n = nU + nI */
  float* LE[YR_NGCF_MAX_LAYERS];      /* saved L E_l */
  float* G[YR_NGCF_MAX_LAYERS + 1];   /* dLoss/dE_l */
  float* T;                           /* [n x d] scratch */
  float *W1[YR_NGCF_MAX_LAYERS], *W2[YR_NGCF_MAX_LAYERS];      /* [d x d] nn.Linear weights */
  float *dW1[YR_NGCF_MAX_LAYERS], *dW2[YR_NGCF_MAX_LAYERS];
  float *mE, *vE;                                              /* Adam moments (NULL for SGD) */
  float *mW1[YR_NGCF_MAX_LAYERS], *vW1[YR_NGCF_MAX_LAYERS], *mW2[YR_NGCF_MAX_LAYERS], *vW2[YR_NGCF_MAX_LAYERS];
  const float* const* E_dev;          /* device copy of E[0..n_layers] */
  float* const* G_dev;                /* device copy of G[0..n_layers] */
  void* ws; size_t ws_bytes;          /* >= yr_ngcf_layer_bwd_ws_bytes(d) */
  double* loss;                       /* device double[2]: [0] running sum of batch means, [1] scratch (zero) */
  int32_t* err;
  /* optional scratch for the row-sparse top-layer backward of yr_ngcf_train_step (all NULL/0 = dense everywhere):
   * row_flag [n] and row_count [1] zero between steps, row_list [row_list_cap], row_list_cap >= 3 * B */
  int32_t* row_flag; int32_t* row_list; int32_t* row_count; int64_t row_list_cap;
  int32_t dense_mode;                 /* yr_dense_mode of this trainer's layers */
  int32_t top_rows_mode;              /* yr_ngcf_train_step, top layer: 1 = backward on the batch rows only (dLoss/dE_L is zero
                                         elsewhere) with G += L^T T as a scatter from those rows; 0 = the dense layer backward.
                                         Same sums, different fp32 order. */
} yr_ngcf_state;

/* forward only: fills E[1..n_layers] (and LE[]) — used by validate / evaluate (propagate ONCE, not per user) */
int yr_ngcf_propagate(const yr_ngcf_state* st, float slope, yr_stream stream);
int yr_ngcf_train_step(const yr_ngcf_state* st, const yr_opt* opt, float slope,
                       const int64_t* uid, const int64_t* pos, const int64_t* neg, int64_t B,
                       float* step_loss, yr_stream stream);
/* The first n_prefix layers of the propagation do not depend on the batch, only on the parameters: a caller that has
 * to read the loss back after every step (train.py does) can enqueue them for the NEXT step with
 * yr_ngcf_propagate_prefix right after the loss copy, so the GPU works through them while the host handles the
 * read-back and stages the next batch, and then passes prefix_done = n_prefix to yr_ngcf_train_step_ex, which starts
 * the forward at that layer. The caller guarantees that no parameter changed in between. prefix_done = 0 is
 * yr_ngcf_train_step. */
int yr_ngcf_propagate_prefix(const yr_ngcf_state* st, float slope, int n_prefix, yr_stream stream);
int yr_ngcf_train_step_ex(const yr_ngcf_state* st, const yr_opt* opt, float slope,
                          const int64_t* uid, const int64_t* pos, const int64_t* neg, int64_t B,
                          float* step_loss, int prefix_done, yr_stream stream);
/* out[r, l*d + k] = E_l[r, k]: the concatenation torch.concat(..., dim=1) of models/ngcf.py:41-43. */
int yr_ngcf_concat(const float* const* E_layers, int n_layers, int64_t n, int d, float* out, yr_stream stream);

/* ---- Laplacian / CSR builder (SURVEY.md 8(f)3) --------------------------------------------------------------
 * NGCFDataPipeline._set_laplacian_matrix (data/datasets/ngcf_data_pipeline.py:19-44) without the two dense
 * (U+I)^2 arrays: interactions (user, item, rating), any order, duplicates averaged (pivot_table mean), zero means
 * dropped -> CSR of L = (D^-1/2 A) D^-1/2 over N = U+I nodes, columns sorted inside a row, fp32 with the reference's
 * association and its row-by-row degree accumulation. rowptr [N+1], col / val [2*nnz] (rowptr[N] entries are used).
 * ws: yr_laplacian_ws_bytes. *err = 1 if an id is out of range (the interaction is skipped). */
size_t yr_laplacian_ws_bytes(int64_t nnz, int64_t num_users, int64_t num_items);
int yr_laplacian_build(const int64_t* user, const int64_t* item, const float* rating, int64_t nnz,
                       int64_t num_users, int64_t num_items, int32_t* rowptr, int32_t* col, float* val,
                       void* ws, size_t ws_bytes, int32_t* err, yr_stream stream);

/* ---- Per-user random split (SURVEY.md 8(f)3) ------------------------------------------------------------------------
 * MFDataPipeline.split (data/datasets/mf_data_pipeline.py:18-52), the pairwise branch: per user
 * train_test_split(test_size=.2, random_state=seed) then train_test_split(rest, test_size=.25, random_state=seed) —
 * sklearn ShuffleSplit on np.random.RandomState(seed).permutation(n), i.e. MT19937 + the legacy Fisher-Yates shuffle,
 * reproduced on the device (the permutation depends on the list length only: one table row per length).
 * ptr/items: CSR over users of the interactions in DataFrame order (int64 item ids). yr_split_sizes gives the three list
 * lengths per user (the caller scans them into train_ptr / valid_ptr / test_ptr); yr_split_per_user fills the lists in
 * the order the reference's frames hold them. ws: yr_split_ws_bytes(max list length). *err = 1: internal stream too
 * short (does not happen with that sizing). */
size_t yr_split_ws_bytes(int max_list_len);
int yr_split_sizes(const int32_t* ptr, int64_t num_users, int32_t* n_train, int32_t* n_valid, int32_t* n_test, yr_stream stream);
int yr_split_per_user(const int32_t* ptr, const int64_t* items, int64_t num_users, int max_list_len, uint32_t seed,
                      const int32_t* train_ptr, const int32_t* valid_ptr, const int32_t* test_ptr,
                      int64_t* train_items, int64_t* valid_items, int64_t* test_items, void* ws, size_t ws_bytes,
                      int32_t* err, yr_stream stream);

/* ---- Scaled synthetic graph (BASELINE config 5, SURVEY.md 8(d)) ------------------------------------------------------
 * The reference has no generator (it reads Yelp's review.json); this is the input producer of the scaled benchmark.
 * yr_synth_user_rows: for every user u the SORTED, DUPLICATE-FREE item list of a synthetic bipartite graph: the number of
 * draws is log-normal (exp(mu + sigma z), clipped to [min_deg, max_deg <= 1024]), every draw is an item rank from a
 * Zipf(zipf_alpha) law mapped to an id by a fixed permutation. Philox4x32-10 streams keyed by (seed, user): the same graph
 * on every rank. Two calls: rowptr == NULL -> cnt_out[u] = list length; rowptr given (exclusive scan of the counts) ->
 * items_out[rowptr[u] ..] = the list. */
int yr_synth_user_rows(uint64_t seed, int64_t num_users, int64_t num_items, double zipf_alpha, double mu, double sigma,
                       int32_t min_deg, int32_t max_deg, const int32_t* rowptr, int32_t* cnt_out, int32_t* items_out,
                       yr_stream stream);
/* Values of L = (D^-1/2 A) D^-1/2 for a BINARY adjacency given as CSR structure (any row block of it):
 * val[k] = (dinv[row] * 1) * dinv[col[k]], dinv = 1 / sqrt(deg) in fp32 — data/datasets/ngcf_data_pipeline.py:34-42.
 * row_node[r] (NULL = r) and col_node[k] index the node degrees `deg`. */
int yr_laplacian_binary_values(const int32_t* rowptr, int64_t n_rows, const int32_t* row_node, const int32_t* col_node,
                               const int32_t* deg, float* val, yr_stream stream);

/* ---- Negative sampler (SURVEY.md 8(f)2) -----------------------------------------------------------------
 * MFDataset._negative_sampling (data/datasets/mf_dataset.py:18-22): for every training interaction t one item
 * drawn uniformly from the items NOT in the user's positive list. pos_ptr/pos_idx: CSR of the users' `pos_items`
 * (mf_data_pipeline.py:41-47), item ids sorted ascending inside a user. Stream: Philox4x32-10, key = seed,
 * counter = (offset + t, block, 0) — a function of (seed, global triple index) only, hence identical under any
 * sharding. A triple that finds no negative within max_blocks*4 draws (user has ~every item) gets -1 and sets
 * *err = 2 (the reference would not terminate); an out-of-range uid sets *err = 1. */
int yr_sample_negatives(const int64_t* uid, int64_t n, const int32_t* pos_ptr, const int32_t* pos_idx,
                        int64_t num_users, int64_t num_items, uint64_t seed, uint64_t offset, int max_blocks,
                        int64_t* neg_out, int32_t* err, yr_stream stream);

/* ------------------------------------------------------------------------------------------------
 * Row-sharded BPR-MF (BASELINE config 5): each rank owns a contiguous block of user rows and of item rows
 * (and their optimizer state). One step = gather owned rows -> all-reduce (NCCL, by the caller) -> per-rank slice
 * of triples -> all-gather of the slice gradients (NCCL) -> owner-side update. The library provides the three
 * device-side pieces; the collectives stay with the caller (torch.distributed / NCCL over NVLink).
 * ---------------------------------------------------------------------------------------------- */

/* out[j*out_ld .. +d) = T_local[ids[j] - row0, :] if row0 <= ids[j] < row1, else zeros.  Every id must fall in
 * exactly one rank's [row0,row1), so the SUM all-reduce of `out` over ranks is the exact gather of all rows.
 * ids outside [0, n_rows_global) set *err. */
int yr_shard_gather_rows(const float* T_local, int64_t row0, int64_t row1, int64_t n_rows_global, int d,
                         const int64_t* ids, int64_t n, float* out, int64_t out_ld, int32_t* err, yr_stream stream);

/* R, G: [B x 3 x d] rows of (user, pos, neg) per triple. For triples b in [b0,b1): x = u.p - u.n, the BPR loss term
 * is added to *loss_acc (sum, not mean) and G[b] = (g*(p-n), g*u, -g*u) with g = -sigmoid(-x)/B (mean over the GLOBAL
 * batch B). Triples outside [b0,b1) are not touched. */
int yr_bpr_rows_grad(const float* R, int d, int64_t B, int64_t b0, int64_t b1, float* G, double* loss_acc,
                     yr_stream stream);

/* Owner-side update of one table shard, in two calls so that several id lists (pos and neg items) feed ONE optimizer
 * step: yr_shard_accumulate adds the gradient rows G[j*g_ld .. +d) of every j with row0 <= ids[j] < row1 into the shard's
 * scratch (duplicates summed); yr_shard_step then performs one optimizer step per row with torch's dense semantics
 * over the shard (SGD with wd = 0 touches only the accumulated rows; max_rows >= number of accumulated ids sizes its
 * grid). gscratch [rows_local x d], flags [rows_local] and counters (>= 64 bytes) must be all-zero on first use and
 * are all-zero again after yr_shard_step; rows_list needs one entry per accumulated id. */
typedef struct yr_shard_state {
  float* T;            /* [rows_local x d] parameters of this shard */
  float *m, *v;        /* Adam moments (NULL for SGD) */
  float* gscratch;
  int32_t* flags;
  int32_t* rows_list;
  int32_t* counters;
  int64_t row0, row1;
  int32_t d;
} yr_shard_state;
int yr_shard_accumulate(const yr_shard_state* st, const yr_opt* opt, const int64_t* ids, int64_t n, const float* G,
                        int64_t g_ld, yr_stream stream);
int yr_shard_step(const yr_shard_state* st, const yr_opt* opt, int64_t max_rows, yr_stream stream);

/* Packed gather for the all-to-all form of the exchange: out[j*out_ld ..] = (sel[j] ? T1 : T0)[row[j], :] — an owner collects,
 * in slot order, the rows of its user-table shard (sel 0) and item-table shard (sel 1) that a requester's slice needs. The
 * caller guarantees row[j] is inside the selected shard. */
int yr_shard_gather_local(const float* T0, const float* T1, int d, const int32_t* sel, const int32_t* row, int64_t n,
                          float* out, int64_t out_ld, yr_stream stream);

/* Ordered (atomics-free) form of yr_shard_accumulate: the caller has grouped the n received gradient rows by local row with
 * a STABLE sort — rows_sorted[j] = local row (ascending), src[j] = index of that gradient row in G — and one warp per
 * segment sums it left to right (arrival order: requester rank, then slot) into the row's scratch. Bit-identical run to
 * run. Entries with rows_sorted[j] < 0 are ignored (gradient rows another shard owns). list_rows != 0 also lists the rows
 * for a sparse step (plain SGD, sparse Adam). */
int yr_shard_accumulate_sorted(const yr_shard_state* st, const yr_opt* opt, const int32_t* rows_sorted, const int32_t* src,
                               int64_t n, const float* G, int64_t g_ld, int list_rows, yr_stream stream);

/* Sparse-traffic ("catch-up") Adam / AdamW for a shard: torch's optimizer is dense (a row without a gradient keeps moving
 * while its moments are non-zero, trainers/base_trainer.py:34-40), but such a row follows a fixed recurrence, so only the
 * rows of the batch are visited: before they are gathered for the forward pass they replay the steps they missed
 * (yr_shard_catch_up: last[row] + 1 .. step - 1, g = 0, the same update code and scalars as the dense sweep), and the rows
 * listed by yr_shard_accumulate_sorted then take step opt->step with their gradient. Bit-identical to
 * yr_shard_step's sweep. scal: 2 * n_scal_steps floats from yr_adam_scalars; last: int32 per local row, zero on first
 * use. flush != 0 brings EVERY row up to opt->step (before the tables are read: evaluation, state_dict). */
int yr_adam_scalars(const yr_opt* opt, int n_steps, float* scal, yr_stream stream);
/* Rows that are about to be READ for the forward pass of step opt->step (rows_sorted: ascending local rows, duplicates
 * allowed) are first brought up to step opt->step - 1. */
int yr_shard_catch_up(const yr_shard_state* st, const yr_opt* opt, const float* scal, int32_t n_scal_steps, int32_t* last,
                      const int32_t* rows_sorted, int64_t n, yr_stream stream);
int yr_shard_step_sparse_adam(const yr_shard_state* st, const yr_opt* opt, const float* scal, int32_t n_scal_steps,
                              int32_t* last, int64_t max_rows, int flush, yr_stream stream);

/* ------------------------------------------------------------------------------------------------
 * CDAE  (models/cdae.py, loss.py:7-16 NSBCELoss, trainers/cdae_trainer.py) — BASELINE config 4
 * ---------------------------------------------------------------------------------------------- */

/* Parameters in the reference's own layouts (state_dict keys hidden_layer.{weight,bias}, user_nodes.weight,
 * output_layer.{weight,bias}); the same struct describes gradients and Adam moments. */
typedef struct yr_cdae_tensors {
  float* Wh;   /* hidden_layer.weight [h x nI]  */
  float* bh;   /* hidden_layer.bias   [h]       */
  float* Vu;   /* user_nodes.weight   [nU x h]  */
  float* Wo;   /* output_layer.weight [nI x h]  */
  float* bo;   /* output_layer.bias   [nI]      */
} yr_cdae_tensors;

size_t yr_cdae_ws_bytes(int64_t B, int64_t nI);

/* BaseModel._activation_module (models/base_model.py:10-14): the two names the reference knows. */
enum yr_activation { YR_ACT_SIGMOID = 0, YR_ACT_IDENTITY = 1 };

/* z[b,:] = sigmoid( Wh . (x[b,:] * keep[b,:]) + bh + Vu[uid[b]] )   (models/cdae.py:46-51; keep == NULL in eval
 * mode, else the dropout multiplier 0 or 1/(1-p) the caller drew — nn.Dropout's mask is supplied, not re-drawn).
 * x is the dense [B x nI] multi-hot `input_mask` exactly as the reference's DataLoader yields it.
 * z_out is [B x ldz] (ldz >= h): columns h..ldz-1 are set to 1, 0, 0, ... so that [z | 1] . [Wo | bo]^T is the
 * output logit (used to feed the full-catalog top-K kernels). */
int yr_cdae_hidden(const yr_cdae_tensors* P, int64_t nU, int64_t nI, int h, const int64_t* uid, const float* x,
                   const float* keep, int64_t B, float* z_out, int64_t ldz, void* ws, size_t ws_bytes,
                   int32_t* err, yr_stream stream);
/* Same with cfg.hidden_activation given (yr_activation; the plain call is sigmoid). h = cfg.hidden_size must be one of
 * 32, 64, 128, 256, 512, 1024 (the values of the reference's cdae_sweep_config.yaml), YR_ERR_BAD_DIM otherwise. */
int yr_cdae_hidden_ex(const yr_cdae_tensors* P, int64_t nU, int64_t nI, int h, int hidden_act, const int64_t* uid,
                      const float* x, const float* keep, int64_t B, float* z_out, int64_t ldz, void* ws, size_t ws_bytes,
                      int32_t* err, yr_stream stream);

/* The hidden activations of yr_cdae_hidden_ex (keep == NULL) from interaction lists instead of a dense multi-hot:
 * z[b, 0:h] = act(bh + Vu[u] + sum over j in in_idx[in_ptr[u] .. in_ptr[u + 1]) of Wh[:, j]), u = user_ids[b]. The lists are
 * a CSR indexed by user id (nU + 1 offsets, ascending unique item ids per row) and Wh is read in place; nothing of size
 * B x nI is needed. Bit-identical to yr_cdae_hidden_ex on the dense multi-hot of the same lists. Columns h..ldz-1 of z
 * are not written. A user id outside [0, nU) sets *err |= 1 and the row is computed for user 0; an item id outside
 * [0, nI), or offsets that decrease or run past in_ptr[nU], set *err |= 2 and the row is computed from an empty list.
 * Nothing is read out of bounds. h as yr_cdae_hidden_ex. */
int yr_cdae_encode(const yr_cdae_tensors* P, int64_t nU, int64_t nI, int h, int hidden_act, const int64_t* user_ids,
                   int64_t B, const int32_t* in_ptr, const int32_t* in_idx, float* z, int64_t ldz, int32_t* err,
                   yr_stream stream);

/* pred[b,i] = sigmoid( z[b,:] . Wo[i,:] + bo[i] )  — CDAE.forward's dense output (models/cdae.py:52). */
int yr_cdae_output(const yr_cdae_tensors* P, int64_t nI, int h, const float* z, int64_t ldz, int64_t B,
                   float* pred, yr_stream stream);

/* One CDAETrainer.train step (trainers/cdae_trainer.py:39-52) or, with opt == NULL, the loss-only pass of
 * validate (:62-70): forward, NSBCELoss over the positions where target + negative_mask != 0 (loss.py:12-16, BCE
 * mean, logs clamped at -100 like torch), backward restricted to those positions with torch's autograd chain
 * d loss / d logit = (p - t) / max((1 - p) p, 1e-12) / m * (1 - p) p (m loss positions; p - t except where p
 * saturates), dense optimizer step over all five tensors. grads must be all-zero on entry and are all-zero on exit.
 * loss (device double[2]): [0] += batch loss, [1] scratch. step_loss may be NULL. `target` is input_mask for train,
 * input_mask + valid_mask for validate. P->Wo and grads->Wo must be aligned to 4 * min(h / 32, 4) bytes (their rows are
 * read and accumulated as float2 / float4), YR_ERR_BAD_ARG otherwise; the other tensors need 4 bytes. */
int yr_cdae_step(const yr_cdae_tensors* P, const yr_cdae_tensors* grads, const yr_cdae_tensors* m,
                 const yr_cdae_tensors* v, const yr_opt* opt, int64_t nU, int64_t nI, int h,
                 const int64_t* uid, const float* x, const float* keep, const float* target,
                 const float* negative_mask, int64_t B, double* loss, float* step_loss,
                 void* ws, size_t ws_bytes, int32_t* err, yr_stream stream);
/* Same with cfg.hidden_activation given (the output activation stays sigmoid: NSBCELoss needs probabilities). */
int yr_cdae_step_ex(const yr_cdae_tensors* P, const yr_cdae_tensors* grads, const yr_cdae_tensors* m,
                    const yr_cdae_tensors* v, const yr_opt* opt, int64_t nU, int64_t nI, int h, int hidden_act,
                    const int64_t* uid, const float* x, const float* keep, const float* target,
                    const float* negative_mask, int64_t B, double* loss, float* step_loss,
                    void* ws, size_t ws_bytes, int32_t* err, yr_stream stream);

/* The same step from INDEX LISTS instead of dense [B x nI] masks (the dense rows the reference's CDAEDataset yields are 152 KB
 * per user; the lists are a few hundred bytes): in_ptr [B + 1] / in_idx = the active inputs of every row (ascending item ids),
 * in_val = their values after dropout (NULL = 1: evaluation), tgt_ptr / tgt_idx / tgt_val = the loss positions of every row
 * (ascending item ids: the union of the target items, value 1, and the sampled negatives, value 0). Same arithmetic and
 * order as yr_cdae_step_ex on the equivalent dense tensors when in_val is NULL or has no zero. A listed input of value 0
 * (dropped by dropout) stays in the hidden layer's sums, where the dense path compacts it out, so the terms are split
 * differently over the partial sums and the results may differ in the last bits. opt == NULL: loss only. */
int yr_cdae_step_idx(const yr_cdae_tensors* P, const yr_cdae_tensors* grads, const yr_cdae_tensors* m,
                     const yr_cdae_tensors* v, const yr_opt* opt, int64_t nU, int64_t nI, int h, int hidden_act,
                     const int64_t* uid, const int32_t* in_ptr, const int32_t* in_idx, const float* in_val,
                     const int32_t* tgt_ptr, const int32_t* tgt_idx, const float* tgt_val, int64_t B,
                     double* loss, float* step_loss, void* ws, size_t ws_bytes, int32_t* err, yr_stream stream);

/* NSBCELoss.forward on dense tensors (loss.py:12-16): mean BCE over positions where target + negative_mask != 0. */
int yr_nsbce_loss(const float* pred, const float* target, const float* negative_mask, int64_t n, float* loss,
                  void* ws, size_t ws_bytes, yr_stream stream);

/* ------------------------------------------------------------------------------------------------
 * Full-catalog evaluation (trainers/mf_trainer.py:134-178, metric.py)
 * ---------------------------------------------------------------------------------------------- */

/* Vt[k, i] = V[i, k] for i < nI; Vt is [d x ldt], ldt >= nI (padding columns are zero-filled). */
int yr_transpose_items(const float* V, int64_t nI, int d, float* Vt, int64_t ldt, yr_stream stream);

/* Workspace of yr_eval_topk_metrics: 256 bytes while the [pad32(d) x 128 users] tile fits shared memory (d up to 288 at
 * K = 10); wider tables keep the tail of the transposed user tile here ((pad32(d) - resident rows) x round_up(n_eval, 128)
 * floats). Any d that is a multiple of 4 is accepted. */
size_t yr_eval_ws_bytes(int64_t n_eval, int d, int K);

/* MFTrainer.evaluate / NGCFTrainer.evaluate fused: for eval row e (user eval_uid[e]) score every item
 * (one fp32 fma chain over k = 0..d-1), overwrite mask_items with -3.40282e+38 (Q4), keep the K best by
 * (score desc, item id asc), then accumulate the reference's metrics (metric.py:7-109, quirks Q6-Q8).
 *   Uemb [nU x d] row-major; Vt [d x ldt] item table transposed (yr_transpose_items);
 *   mask_ptr/mask_idx: CSR over eval rows, item ids ascending per row;
 *   act_ptr/act_idx:  CSR over eval rows, pos_items in their ORIGINAL order; act_nuniq[e] = |set(pos_items)|;
 *   inv_log2 [K] (double) = 1/log2(i+2), host-computed so DCG matches Python's math.log2;
 *   topk_out [n_eval x K] int64 best first; user_metrics [n_eval x 4] double =
 *   (hits/K, hits/|set(A)| or 0, AP, NDCG) per row; metric_sums [6] double =
 *   (sum precision, sum recall, sum AP, sum NDCG, #rows with |set(A)|>0, #rows with len(A)>0).
 * The score matrix is never written to memory. ws: yr_eval_ws_bytes(n_eval, d, K) bytes (YR_ERR_WORKSPACE if smaller). */
int yr_eval_topk_metrics(const float* Uemb, int64_t nU, const float* Vt, int64_t ldt, int64_t nI, int d,
                         const int64_t* eval_uid, int64_t n_eval,
                         const int32_t* mask_ptr, const int32_t* mask_idx,
                         const int32_t* act_ptr, const int32_t* act_idx, const int32_t* act_nuniq,
                         const double* inv_log2, int K,
                         int64_t* topk_out, float* topk_score, double* user_metrics, double* metric_sums,
                         void* ws, size_t ws_bytes, int32_t* err, yr_stream stream);

/* Same contract and BIT-IDENTICAL outputs as yr_eval_topk_metrics, on the tensor cores: TF32 tcgen05.mma scores
 * act as a candidate filter with a proven error bound (|s_tf32 - s_fp32| <= c * ||u|| * max||v||), the few survivors
 * per row are re-scored with the canonical fp32 fma chain, and rows the filter cannot decide (more than 32 items
 * inside the window, or fewer than K unmasked items) are evaluated by the exact kernel. Needs both layouts of the
 * item table: Vemb [nI x d] row-major (TMA source, exact re-score) and Vt (yr_transpose_items, for the fallback).
 * Supported when yr_eval_tc_supported(d, K) != 0 (d % 32 == 0, 32 <= d <= 256, K <= 16); otherwise YR_ERR_BAD_DIM
 * and the caller uses yr_eval_topk_metrics. ws: yr_eval_tc_ws_bytes(n_eval) bytes. */
int yr_eval_tc_supported(int d, int K);
size_t yr_eval_tc_ws_bytes(int64_t n_eval);
int yr_eval_topk_metrics_tc(const float* Uemb, int64_t nU, const float* Vemb, const float* Vt, int64_t ldt,
                            int64_t nI, int d, const int64_t* eval_uid, int64_t n_eval,
                            const int32_t* mask_ptr, const int32_t* mask_idx,
                            const int32_t* act_ptr, const int32_t* act_idx, const int32_t* act_nuniq,
                            const double* inv_log2, int K,
                            int64_t* topk_out, float* topk_score, double* user_metrics, double* metric_sums,
                            void* ws, size_t ws_bytes, int32_t* err, yr_stream stream);

/* MFTrainer._generate_top_k_recommendation (trainers/mf_trainer.py:163-178) for ONE score row:
 * mask_idx (int64, any order, n_mask entries) positions get -3.40282e+38, then the K best by
 * (score desc, item id asc) are written best-first. `pred` is not modified. */
int yr_topk_masked_row(const float* pred, int64_t nI, const int64_t* mask_idx, int64_t n_mask, int K,
                       int64_t* topk_out, yr_stream stream);

/* The same for a batch of score rows of ANY model — the device half of DCN's chunked evaluator
 * (trainers/dcn_trainer.py:145-203, :188-203): pred [n_rows x ld] holds one full-catalog score row per evaluated user
 * (assembled chunk by chunk by the caller's model), mask CSR (int32, ids in [0, nI)) per row, masked positions take
 * `mask_value` (DCN: 0, its outputs are sigmoids; MF / NGCF: -3.40282e+38), K best by (score desc, item id asc) per row.
 * ws: n_rows * nI bytes. */
int yr_topk_masked_rows(const float* pred, int64_t ld, int64_t n_rows, int64_t nI, const int32_t* mask_ptr,
                        const int32_t* mask_idx, float mask_value, int K, int64_t* topk_out, void* ws, size_t ws_bytes,
                        yr_stream stream);

/* One item slice of an item-sliced evaluation: yr_eval_topk_metrics_tc on items [i0, i0 + nI) of the catalog (Vemb / Vt point
 * at the slice, mask lists hold slice-local ids) as call `slice` of `n_slices` concurrent calls (one stream each) that share
 * xchg [n_slices x n_eval] floats (-inf on entry): every call publishes its running lower bound of each row's K-th best score
 * there and reads the others', so no slice pays the warm-up of a threshold of its own. topk_out / topk_score [n_eval x K]
 * receive the slice's survivors (slice-local ids, exact scores; lists shorter than K are padded with id -1 / -inf);
 * user_metrics / metric_sums are not written for n_slices > 1. yr_topk_merge + yr_topk_metrics finish the evaluation. */
int yr_eval_topk_metrics_tc_slice(const float* Uemb, int64_t nU, const float* Vemb, const float* Vt, int64_t ldt, int64_t nI,
                                  int d, const int64_t* eval_uid, int64_t n_eval, const int32_t* mask_ptr,
                                  const int32_t* mask_idx, const int32_t* act_ptr, const int32_t* act_idx,
                                  const int32_t* act_nuniq, const double* inv_log2, int K, int64_t* topk_out,
                                  float* topk_score, double* user_metrics, double* metric_sums, void* ws, size_t ws_bytes,
                                  int32_t* err, int slice, int n_slices, float* xchg, yr_stream stream);

/* Item-sliced evaluation (small row shards: a shard of 31 user tiles cannot fill 148 SMs, so the catalog is cut into S
 * disjoint item slices that are evaluated by S concurrent yr_eval_topk_metrics_tc_slice calls): merges the
 * per-slice lists ids / scores [S x n x K] (slice-local ids, exact scores, id -1 = padding) into the K best per row by
 * (score desc, global id = id + id_offset[slice] asc) — the same lists, in the same order, as the unsliced call
 * (trainers/mf_trainer.py:163-178 semantics). S * K <= 64. out_scores may be NULL. */
int yr_topk_merge(const int64_t* ids, const float* scores, int S, int64_t n, int K, const int64_t* id_offset,
                  int64_t* out_ids, float* out_scores, yr_stream stream);

/* metric.py:7-109 on device for already-computed recommendations: predicted [n x ldp] int64 (first K columns
 * used), actual as CSR in original order. Same outputs as yr_eval_topk_metrics. */
int yr_topk_metrics(const int64_t* predicted, int64_t ldp, int64_t n, const int32_t* act_ptr,
                    const int32_t* act_idx, const int32_t* act_nuniq, const double* inv_log2, int K,
                    double* user_metrics, double* metric_sums, yr_stream stream);

/* ----------------------------------------------------------------------------------------------
 * Top-K retrieval (retrieval.cu)
 * ---------------------------------------------------------------------------------------------- */
enum yr_dtype { YR_DTYPE_F32 = 0, YR_DTYPE_BF16 = 1 };

/* For each of the B users user_ids[b]: score = U[uid] . V[i] over all nI items (U [nU x d], V [nI x d], both row-major
 * of `dtype`, fp32 accumulation in one fma chain per score, k ascending: the scores of yr_eval_topk_metrics), and
 * out_ids / out_scores [B x K] = the K best items by (score desc, item id asc). The B x nI scores are never stored.
 * seen_ptr / seen_idx (both NULL = no seen lists): CSR of seen items, ascending per row, indexed by the user id
 * (seen_by_row = 0, nU + 1 offsets) or by the batch row b (seen_by_row = 1, B + 1 offsets). A seen item scores
 * masked_score instead: -INFINITY excludes it. Items scoring -inf or NaN are never returned; a row with fewer than K
 * returnable items is padded with id -1 / score -inf. A user id outside [0, nU) sets *err = 1 (err may be NULL) and
 * gets an all-padding row. 1 <= K <= 1024, d % 8 == 0, d <= 1024, nI < 2^31 - 1.
 * ws: yr_recommend_ws_bytes(B, nI, K) bytes (0 = none needed; same device as the call). */
size_t yr_recommend_ws_bytes(int64_t B, int64_t nI, int K);
int yr_recommend_topk(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype, const int64_t* user_ids,
                      int64_t B, const int32_t* seen_ptr, const int32_t* seen_idx, int seen_by_row, float masked_score,
                      int K, int64_t* out_ids, float* out_scores, void* ws, size_t ws_bytes, int32_t* err,
                      yr_stream stream);
/* Same with a per-item bias: item_bias [nI] fp32 (for fp32 and bf16 tables; NULL = none) makes the score
 * U[uid] . V[i] + item_bias[i], the bias added after the fma chain, before seen items are masked. That equals, bit for bit,
 * the unbiased call on the tables [U | 1 | 0...] and [V | item_bias | 0...]. */
int yr_recommend_topk_ex(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype, const int64_t* user_ids,
                         int64_t B, const int32_t* seen_ptr, const int32_t* seen_idx, int seen_by_row, float masked_score,
                         int K, int64_t* out_ids, float* out_scores, void* ws, size_t ws_bytes, int32_t* err,
                         yr_stream stream, const float* item_bias);

/* yr_recommend_topk restricted per row to one subset of the catalog. The G subsets are a CSR of item ids: subset g is
 * subset_idx[subset_ptr[g] .. subset_ptr[g + 1]), ascending and duplicate-free; subsets may overlap. Row b ranks only the
 * items of subset subset_ids[b], or the whole catalog when subset_ids[b] = -1, and gets exactly the ids and scores
 * yr_recommend_topk returns when every other item is a seen item with masked_score = -INFINITY (same scores, order,
 * seen-item exclusion via seen_ptr / seen_idx indexed by user id, padding with id -1 / score -inf). Rows are grouped by
 * subset on the device; outputs are in request order. max_subset_len: the longest list a row streams (the longest
 * subset, nI if a row is -1); it only sets the number of item splits, any value >= 0 gives the same results. A user id
 * outside [0, nU) sets bit 0 of *err (*err |= 1), a subset id outside [-1, G) bit 1 (*err |= 2); either row is all
 * padding. B < 2^31 - 1, G >= 0; the other limits as yr_recommend_topk.
 * ws: yr_recommend_subset_ws_bytes(B, G, max_subset_len, K) bytes (row grouping and per-split lists; same device). */
size_t yr_recommend_subset_ws_bytes(int64_t B, int G, int64_t max_subset_len, int K);
int yr_recommend_subset_topk(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype,
                             const int64_t* user_ids, int64_t B, const int32_t* subset_ptr, const int32_t* subset_idx,
                             int G, int64_t max_subset_len, const int64_t* subset_ids, const int32_t* seen_ptr,
                             const int32_t* seen_idx, int K, int64_t* out_ids, float* out_scores, void* ws,
                             size_t ws_bytes, int32_t* err, yr_stream stream);
/* Same with a per-item bias, as yr_recommend_topk_ex. */
int yr_recommend_subset_topk_ex(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype,
                                const int64_t* user_ids, int64_t B, const int32_t* subset_ptr, const int32_t* subset_idx,
                                int G, int64_t max_subset_len, const int64_t* subset_ids, const int32_t* seen_ptr,
                                const int32_t* seen_idx, int K, int64_t* out_ids, float* out_scores, void* ws,
                                size_t ws_bytes, int32_t* err, yr_stream stream, const float* item_bias);

/* yr_recommend_topk_ex restricted per row to the items within a radius of a point on the sphere. Item i is inside row b
 * iff ((c_x * p_x) + (c_y * p_y)) + (c_z * p_z) >= threshold[b] in float64, each product and sum rounded on its own,
 * where c = centre_xyz[3b .. 3b + 3) is the centre's unit vector, p = item_xyz[3i .. 3i + 3) the item's, and
 * threshold[b] = cos(radius / Earth radius) (-INFINITY: every item). Row b gets exactly the ids and scores
 * yr_recommend_topk_ex returns when every item outside is a seen item with masked_score = -INFINITY (seen lists indexed
 * by user id; item_bias may be NULL). The item grid: cells of cell_deg degrees, num_lat = ceil(180 / cell_deg) lat bands
 * and num_lon = ceil(360 / cell_deg) lon bands; an item at (lat, lon) degrees is in band floor((lat + 90) / cell_deg)
 * and floor((lon + 180) / cell_deg), each clamped to the grid, cell key = lat band * num_lon + lon band. cell_items
 * [nI] holds the item ids sorted by (key, id), cell_keys [num_cells] the ascending keys of the non-empty cells and
 * cell_ptr [num_cells + 1] their offsets into cell_items. The grid only bounds which items are read: results do not
 * depend on it as long as item_xyz and the cells come from the same (lat, lon). A user id outside [0, nU) sets
 * *err |= 1, a non-finite centre or a NaN / +inf threshold *err |= 2; either row is all padding. The number of item
 * splits follows nI (no device read). Other limits as yr_recommend_subset_topk.
 * ws: yr_recommend_geo_ws_bytes(B, nI, K) bytes (window and row grouping per request, per-split lists; same device). */
size_t yr_recommend_geo_ws_bytes(int64_t B, int64_t nI, int K);
int yr_recommend_geo_topk(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype, const int64_t* user_ids,
                          int64_t B, const int64_t* cell_keys, const int32_t* cell_ptr, int64_t num_cells,
                          const int32_t* cell_items, const double* item_xyz, double cell_deg, int64_t num_lat,
                          int64_t num_lon, const double* centre_xyz, const double* threshold, const int32_t* seen_ptr,
                          const int32_t* seen_idx, int K, int64_t* out_ids, float* out_scores, void* ws, size_t ws_bytes,
                          int32_t* err, yr_stream stream, const float* item_bias);

/* Diversity re-ranking (Maximal Marginal Relevance) of B pools of N candidates, e.g. the output of yr_recommend_topk
 * with K = N. Position j of row b holds item p_j = pool_ids[b * N + j] (-1: an empty slot) with relevance
 * r_j = pool_scores[b * N + j]. V [nI x d] of `dtype` is the item table similarity is measured in. With fp32 arithmetic,
 * every operation separately rounded (no fma contraction outside the sums):
 *   ss_j = sum_k V[p_j,k]^2 (any summation order), n_j = 1 / sqrt(ss_j) (sqrt and reciprocal each correctly rounded;
 *   n_j = 0 when ss_j == 0), sim(i, j) = dot(V[p_i], V[p_j]) * (n_i * n_j) (the dot in any summation order).
 * a = lam and c = one_minus_lam, both computed by the caller (c = fl(1 - a)). For t = 0 .. K-1: pen_j = 0 while nothing
 * has been picked, after that the maximum of sim(j, s) over the picked positions s (a NaN similarity makes it NaN);
 * m_j = (a * r_j) - (c * pen_j), with -0 ranking as +0 and NaN as -inf. Step t picks the unpicked non-empty position
 * with the largest m_j, ties to the lower position, and writes out_ids[b * K + t] = p_j and out_scores[b * K + t] = r_j
 * (pick order; the scores stay the pool's). When no non-empty position is left the rest of the row is -1 / -INFINITY.
 * With lam = 1 and finite similarities, m_j = r_j: a pool in (score desc, id asc) order, as yr_recommend_topk writes
 * it, comes back as its first K entries. A pool id outside [-1, nI) sets *err |= 1 (err may be
 * NULL) and makes the row all padding. 1 <= K <= N <= 1024, 0 <= lam, one_minus_lam <= 1, d % 8 == 0, d <= 1024,
 * nI < 2^31 - 1, B < 2^31 - 1. No workspace. */
int yr_recommend_mmr(const void* V, int64_t nI, int d, int dtype, const int64_t* pool_ids, const float* pool_scores,
                     int64_t B, int N, int K, float lam, float one_minus_lam, int64_t* out_ids, float* out_scores,
                     int32_t* err, yr_stream stream);

/* Group retrieval: one ranked list for each of G groups of users. Group g has the m_g members
 * members[group_ptr[g] .. group_ptr[g + 1]) (rows of U), 1 <= m_g <= YR_GROUP_MAX_MEMBERS; the caller lists them in
 * ascending order without duplicates (retrieval.UserGroups does). For item i, s_j(i) is exactly the score
 * yr_recommend_topk_ex gives member j (one fp32 fma chain, k ascending, then + item_bias[i] if item_bias is not NULL),
 * and the group's score is
 *   agg = YR_GROUP_MIN (least misery): a(i) = min_j s_j(i), NaN if any s_j(i) is NaN;
 *   agg = YR_GROUP_MEAN: S = (((s_1 + s_2) + s_3) + ...) in member order, each add rounded on its own, then
 *                        a(i) = S / m_g, one correctly rounded division.
 * An item in the seen list of any member (seen_ptr / seen_idx indexed by the member's row of U; both NULL = none) is
 * never returned; nor is an item scoring -inf or NaN. Ranking, ties and padding as yr_recommend_topk: out_ids /
 * out_scores [G x K] by (a desc, id asc), short rows padded with id -1 / score -inf, rows in request order. A group of
 * one member u gets exactly yr_recommend_topk_ex's row for u. subset_ids (NULL = every group ranks the whole catalog)
 * restricts group g to subset subset_ids[g] of the subset CSR (subset_ptr [num_subsets + 1], subset_idx), -1 = the
 * whole catalog, as yr_recommend_subset_topk (max_subset_len as there; with subset_ids NULL it is not read). No buffer
 * of G x nI scores is made. num_members: the length of members. A member outside [0, nU) sets *err |= 1, a subset id
 * outside [-1, num_subsets) *err |= 2, a group size outside [1, YR_GROUP_MAX_MEMBERS] (or a group_ptr range outside
 * members) *err |= 4; each such row is all padding. G < 2^31 - 1; the other limits as yr_recommend_subset_topk.
 * ws: yr_recommend_group_ws_bytes(G, num_subsets, max_subset_len, K) bytes (per-split lists and, with subset_ids, the
 * row grouping; same device); without subset_ids pass num_subsets = 0 and max_subset_len = nI. */
#define YR_GROUP_MAX_MEMBERS 32
enum yr_group_agg { YR_GROUP_MIN = 0, YR_GROUP_MEAN = 1 };
size_t yr_recommend_group_ws_bytes(int64_t G, int num_subsets, int64_t max_subset_len, int K);
int yr_recommend_group_topk(const void* U, int64_t nU, const void* V, int64_t nI, int d, int dtype,
                            const int32_t* group_ptr, int64_t G, const int64_t* members, int64_t num_members, int agg,
                            const int32_t* subset_ptr, const int32_t* subset_idx, int num_subsets,
                            int64_t max_subset_len, const int64_t* subset_ids, const int32_t* seen_ptr,
                            const int32_t* seen_idx, int K, int64_t* out_ids, float* out_scores, void* ws,
                            size_t ws_bytes, int32_t* err, yr_stream stream, const float* item_bias);

#ifdef __cplusplus
}
#endif
#endif /* YELPREC_B200_H */
