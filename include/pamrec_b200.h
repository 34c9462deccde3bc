/*
 * pamrec_b200 — C ABI of the B200-native PAMRec train / score step.
 *
 * This is the drop-in boundary for the reference's device work.  The reference has no
 * FFI: its "device" is a TensorFlow session, and the calls this library replaces are the
 * three `sess.run` sites plus the graph construction they depend on (all paths relative
 * to the reference root, reco_utils/recommender/deeprec/...):
 *
 *   pamrec_train_step   <->  PAMRECModel.train            models/sequential/pamrec.py:426-453
 *                            (update + BN moving stats + 5 loss scalars in one run)
 *   pamrec_forward      <->  SequentialBaseModel.eval_with_user / eval / infer
 *                            models/sequential/sequential_base_model.py:502-516, 415-418, 557-560
 *   pamrec_create/bind  <->  BaseModel.__init__ graph + session bootstrap, models/base_model.py:20-75
 *   PamrecBatch         <->  SequentialIterator.gen_feed_dict, io/sequential_iterator.py:1143-1181
 *   parameter inventory <->  tf.get_variable sites (SURVEY.md Appendix B)
 *
 * Conventions: plain C, no exceptions, int return (0 = ok, <0 = error, text through
 * pamrec_last_error).  The CALLER owns every device buffer (the Python host allocates
 * them with torch); the library owns nothing on the device, never frees caller memory
 * and keeps no hidden global state (one handle per stream / thread).  Every launch goes
 * to the `stream` argument (a cudaStream_t passed as void*).  All tensors are row-major,
 * contiguous; ids are int32, values fp32.
 */
#ifndef PAMREC_B200_H_
#define PAMREC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* PAMRec's embedding widths (also what a sibling model runs with PamrecConfig.item_dim / cate_dim / user_dim = 0) */
#define PAMREC_ITEM_DIM 16
#define PAMREC_CATE_DIM 4
#define PAMREC_USER_DIM 20
#define PAMREC_EMB_DIM 20   /* item + cate */
#define PAMREC_D 40         /* model width = 2 * (item + cate), pamrec.py:144,523 */
#define PAMREC_NBUCKET 10   /* rows of the time-aware Q/K/V tables, pamrec.py:699-713 */
#define PAMREC_GROUP 5      /* listwise group, pamrec.py:73-75 */
#define PAMREC_MAX_T 256

typedef struct PamrecHandle_* PamrecHandle;

/* sparse (embedding-table) Adam flavours, SURVEY.md section 7 H2 */
enum { PAMREC_ADAM_DENSE_EXACT = 0, /* tf.train.AdamOptimizer: decay + update EVERY row     */
       PAMREC_ADAM_LAZY = 1 };      /* touched rows only (tf.contrib.opt.LazyAdamOptimizer) */

/* embedding-table placement */
enum { PAMREC_TABLES_LOCAL = 0,     /* whole tables on this GPU, direct gather (world_size must be 1)          */
       PAMREC_TABLES_SHARDED = 1,   /* row r lives on rank r % world_size at local row r / world_size; rows
                                       and row gradients travel by all-to-all (works with world_size 1 too) */
       PAMREC_TABLES_REPLICATED = 2 }; /* every rank holds whole tables (small vocabularies): direct gather, the merged row
                                       gradients and the looked-up-row marks are all-reduced with the dense gradients
                                       and every rank applies the same update (world_size 1: same as LOCAL)     */

/* model family (all share the feed dict, the tables, BN / clip / Adam semantics and the C ABI below).  The sibling multi-task
 * baselines of the reference (SURVEY.md section 8(f) row N3) run on one GPU with whole tables (PAMREC_TABLES_LOCAL):
 *   PAMREC_MODEL_MMOE         MMoEModel_original   models/sequential/mmoe.py:24-82, 183-337
 *   PAMREC_MODEL_PLE          PLEModel             models/sequential/ple.py:24-60
 *   PAMREC_MODEL_SHAREBOTTOM  ShareBottomModel     models/sequential/sharebottom.py:160-203
 *   PAMREC_MODEL_SASREC       SASRecModel          models/sequential/sasrec.py:16-96, 230-330
 * The first three: DIN-style attention pooling (`_attention_fcn`) of the satisfied-only and of the full history against the target
 * item, a mixing layer (MMoE / PLE / none) and two towers; loss = data + regular + 0.5 * auxiliary.  SASRec: the satisfied-only
 * history + a position table through two 20-wide self-attention blocks with dense Q / K / V, the state at the last satisfied
 * position | target into one tower; loss = data + regular (single task; no user tables: the ulong / ushort buffers are unused). */
enum { PAMREC_MODEL_PAMREC = 0, PAMREC_MODEL_MMOE = 1, PAMREC_MODEL_PLE = 2, PAMREC_MODEL_SHAREBOTTOM = 3, PAMREC_MODEL_SASREC = 4 };

/* hparams.loss */
enum { PAMREC_LOSS_XENT = 0,        /* "cross_entropy_loss" (config/mmoe.yaml)                                  */
       PAMREC_LOSS_SOFTMAX = 1 };   /* "softmax" over groups of train_num_ngs + 1 rows (base_model.py:222-242)  */

typedef struct PamrecConfig {
  int32_t n_users, n_items, n_cates; /* vocabulary sizes = table rows (sequential_base_model.py:565-567) */
  int32_t max_seq_len;               /* T, hparams.max_seq_length                                       */
  int32_t max_batch;                 /* capacity B; training batches must be multiples of PAMREC_GROUP   */
  float learning_rate, beta1, beta2, epsilon; /* tf.train.AdamOptimizer(lr), base_model.py:270-271      */
  float embed_l2, layer_l2;          /* base_model.py:122-134                                           */
  float max_grad_norm;               /* per-tensor tf.clip_by_norm, base_model.py:297-303               */
  int32_t is_clip_norm;
  float fuzhu_weight;                /* pamrec.py:106                                                   */
  float order_weight;                /* hparams.discrepancy_loss_weight, pamrec.py:79                   */
  int32_t sparse_adam_mode;          /* PAMREC_ADAM_*                                                   */
  /* data parallel over listwise groups, one process per GPU (no reference counterpart: the
   * reference is single-device).  Each rank passes its share of one GLOBAL batch; batch-norm
   * statistics, clip norms, loss means and dense gradients are all-reduced inside the step,
   * so the result equals the single-GPU step on the concatenated batch.  world_size > 1
   * needs pamrec_comm_init and table_mode = PAMREC_TABLES_SHARDED or _REPLICATED.         */
  int32_t world_size, rank;
  int32_t table_mode;                /* PAMREC_TABLES_*                                                 */
  /* hparams.loss (base_model.py:195-242, pamrec.py:81-106): PAMREC_LOSS_XENT = "cross_entropy_loss" (mean sigmoid cross
   * entropy, the quick start); PAMREC_LOSS_SOFTMAX = "softmax": -group * mean(log(where(label == 1, softmax over groups of
   * `softmax_group` = train_num_ngs + 1 consecutive logits, 1))) for both the satisfied and the play head.  The order loss
   * (groups of 5) and the L2 term are the same in both.  Batches must then be multiples of softmax_group; with
   * world_size > 1 softmax_group must divide 5 (ranks hold whole listwise groups of 5).                                   */
  int32_t loss_kind;
  int32_t softmax_group;             /* used by PAMREC_LOSS_SOFTMAX only; 0 is read as 1                */
  int32_t model_kind;                /* PAMREC_MODEL_*                                                  */
  /* embedding widths (hparams.item_embedding_dim / cate_embedding_dim / user_embedding_dim); 0 = 16 / 4 / 20 each.  PAMREC_MODEL_PAMREC
   * runs 16 / 4 / 20 only.  The sibling models run (item, cate) = (16, 4) or (32, 8) - the reference's config/ple.yaml,
   * sharebottom.yaml and sasrec.yaml use 32 / 8 - with user = 16, 20 or 40; any other set is refused (pamrec_create returns -10). */
  int32_t item_dim, cate_dim, user_dim;
} PamrecConfig;

/* One batch, device pointers (layouts of io/sequential_iterator.py:1111-1135). */
typedef struct PamrecBatch {
  int32_t batch;                      /* B rows in this batch (<= max_batch)                   */
  const int32_t* item_history;        /* [B,T]                                                 */
  const int32_t* item_cate_history;   /* [B,T]                                                 */
  const float* item_loop_times_history; /* [B,T] play-ratio bucket as float; cast like pamrec.py:716 */
  const int32_t* mask;                /* [B,T] 1 = real position                               */
  const int32_t* users;               /* [B]                                                   */
  const int32_t* items;               /* [B]                                                   */
  const int32_t* cates;               /* [B]                                                   */
  const float* labels_satisfied;      /* [B]  (train only)                                     */
  const float* labels_play;           /* [B]  (train only)                                     */
  const float* plays;                 /* [B]  bucket index as float (train only)               */
  int32_t global_batch;               /* rows of the whole global batch over all ranks; 0 = batch * world_size.
                                         batch may be 0 on a rank that only takes part in the collectives   */
  /* satisfied-only copy of the history, compacted to the left (io/sequential_iterator.py:1069-1103): read by the sibling
   * models only (PAMREC_MODEL_MMOE / _PLE / _SHAREBOTTOM / _SASREC, mmoe.py:199-201, sasrec.py:55-64); may be NULL for PAMREC_MODEL_PAMREC */
  const int32_t* satisfied_item_history; /* [B,T]                                              */
  const int32_t* satisfied_cate_history; /* [B,T]                                              */
  const int32_t* satisfied_mask;         /* [B,T] 1 = real position                            */
} PamrecBatch;

/* Caller-owned device memory handed to the library once. */
typedef struct PamrecBuffers {
  float* dense_param; float* dense_grad; float* dense_m; float* dense_v; /* [dense_numel] each      */
  float* bn_moving;                                                      /* [bn_numel] mean|var sets */
  /* tables: [rows,width] with rows = vocabulary size (PAMREC_TABLES_LOCAL / _REPLICATED) or pamrec_shard_rows (SHARDED) */
  float* item_w; float* item_m; float* item_v;                           /* [rows(n_items),item_dim] */
  float* cate_w; float* cate_m; float* cate_v;                           /* [rows(n_cates),cate_dim] */
  float* ulong_w; float* ulong_m; float* ulong_v;                        /* [rows(n_users),user_dim] */
  float* ushort_w; float* ushort_m; float* ushort_v;                     /* [rows(n_users),user_dim] */
  void* workspace; size_t workspace_bytes;                               /* >= pamrec_workspace_bytes */
} PamrecBuffers;

/* Named slice of one of the caller's pools. */
enum { PAMREC_POOL_DENSE = 0, PAMREC_POOL_BN = 1, PAMREC_POOL_WORKSPACE = 2 };
enum { PAMREC_F32 = 0, PAMREC_I32 = 1, PAMREC_F64 = 2, PAMREC_U8 = 3 };
enum { PAMREC_SEG_L2 = 1,        /* in layer_params: gets layer_l2 (sequential_base_model.py:714-721) */
       PAMREC_SEG_POS = 2,       /* position table: sparse-style clip norm, no L2                     */
       PAMREC_SEG_DEAD = 4 };    /* never reaches the logits: gradient is the L2 term only            */
typedef struct PamrecTensorInfo {
  char name[160];     /* TF variable name (dense / bn pools) or workspace tensor name */
  int32_t pool, dtype, flags;
  int64_t offset;     /* element offset inside the pool (bytes for the workspace pool) */
  int64_t numel;
  int32_t ndim; int64_t shape[4];
} PamrecTensorInfo;

const char* pamrec_version(void);
/* sizeof of the structs of this header as compiled into the library, in the order PamrecConfig, PamrecBatch, PamrecBuffers,
 * PamrecTensorInfo, PamrecLines: lets a foreign-language binding check its mirror of the layouts before the first call */
int pamrec_abi_sizes(int64_t out[6]);

/* Host-only: allowed without a GPU. */
int pamrec_create(const PamrecConfig* cfg, PamrecHandle* out);
int pamrec_destroy(PamrecHandle h);
const char* pamrec_last_error(PamrecHandle h);
int64_t pamrec_dense_numel(PamrecHandle h);
int64_t pamrec_bn_numel(PamrecHandle h);
size_t pamrec_workspace_bytes(PamrecHandle h);
int pamrec_tensor_count(PamrecHandle h, int pool);
int pamrec_tensor_info(PamrecHandle h, int pool, int index, PamrecTensorInfo* out);

/* Device entry points. */
int pamrec_bind(PamrecHandle h, const PamrecBuffers* bufs, void* stream);
/* gather only: x0[B,T,40] = item|cate|target + position (sequential_base_model.py:603-616,666-668; pamrec.py:155-159,251-257) */
int pamrec_gather_fwd(PamrecHandle h, const PamrecBatch* b, float* x0_out, void* stream);
/* forward; training=0 -> BN moving stats (eval_with_user), writes sigmoid(logit) to pred_out[B] if non-null */
int pamrec_forward(PamrecHandle h, const PamrecBatch* b, int training, float* pred_out, void* stream);
/* losses + backward into dense_grad / workspace (requires pamrec_forward(training=1) on the same batch) */
int pamrec_backward(PamrecHandle h, const PamrecBatch* b, void* stream);
/* per-tensor clip + Adam on dense and sparse variables; `step` is 1-based (beta powers).  step = 0 (one GPU, whole tables):
 * use and advance the step counter the library keeps on the device (every call with step >= 1 sets it) - the form to capture
 * in a CUDA graph, where a host-computed step size would be frozen into the captured launch arguments */
int pamrec_apply_gradients(PamrecHandle h, const PamrecBatch* b, int64_t step, void* stream);
/* forward + backward + apply; losses_out (device, 5 floats): loss, data, regular, auxiliary, order (pamrec.py:444-448) */
int pamrec_train_step(PamrecHandle h, const PamrecBatch* b, int64_t step, float* losses_out, void* stream);

/* Multi-GPU plumbing.  The library talks to NCCL directly (dlopen of the libnccl.so.2 that PyTorch ships;
 * `nccl_path` may be NULL to use the loader's search path).  Rank 0 creates the unique id, the host broadcasts
 * the 128 bytes (torch.distributed), every rank calls pamrec_comm_init; afterwards forward / backward /
 * apply_gradients / train_step are collective calls that every rank must make in the same order. */
#define PAMREC_COMM_ID_BYTES 128
int pamrec_comm_unique_id(const char* nccl_path, char id_out[PAMREC_COMM_ID_BYTES]);
int pamrec_comm_init(PamrecHandle h, const char* nccl_path, const char id[PAMREC_COMM_ID_BYTES]);
int pamrec_comm_destroy(PamrecHandle h);
/* Optional peer-memory mailboxes (NVLink P2P, world_size <= 8): with them the persistent head kernels exchange the batch-norm
 * column sums of a train step inside their grid barriers, by stores into their peers' mailboxes, and the gradients are summed
 * through the mailboxes as well; without them NCCL does both.
 * Every rank calls _create, the host all-gathers the 64-byte handles (rank-major), every rank calls _open. */
#define PAMREC_IPC_HANDLE_BYTES 64
int pamrec_comm_mailbox_create(PamrecHandle h, char handle_out[PAMREC_IPC_HANDLE_BYTES]);
int pamrec_comm_mailbox_open(PamrecHandle h, const char* handles);
/* rows of this rank's shard of a table with `vocab_rows` rows: ceil(vocab_rows / world_size) (all ranks equal, tail padded) */
int64_t pamrec_shard_rows(PamrecHandle h, int64_t vocab_rows);
/* sum-all-reduce of a caller buffer over the handle's communicator (dtype PAMREC_F32 / PAMREC_F64 / PAMREC_I32) */
int pamrec_comm_all_reduce(PamrecHandle h, void* dptr, int64_t count, int dtype, void* stream);

/* Stand-alone HBM kernels for roofline measurement (same kernels the step uses). */
int pamrec_bench_gather(PamrecHandle h, const int32_t* item_ids, const int32_t* cate_ids, const int32_t* tgt_items,
                        const int32_t* tgt_cates, int64_t n_rows, int32_t T, float* out, void* stream);
int pamrec_bench_table_adam(PamrecHandle h, int64_t step, void* stream);

/* Test hooks.  PAMREC_DEBUG_SAVE_FFN_HIDDEN: pamrec_forward(training = 1) also stores relu(f W1 + b1) of encoder block 0 / 1 in
 * the workspace tensors "d_Q" / "d_K" (backward-only scratch, overwritten by pamrec_backward), so that a checker can read the
 * exact ReLU pattern of the point-wise FFN (pamrec.py:565-570).  Costs one extra [B,T,40] store per block; off by default. */
#define PAMREC_DEBUG_SAVE_FFN_HIDDEN 1
/* PAMREC_DEBUG_HEAD_TRACE: the persistent head kernels stamp %globaltimer (ns) at their start and at every grid barrier;
 * pamrec_head_trace copies the 32 stamps of the last forward (backward = 0) or backward (1) head kernel: [0 .. n-1] barrier
 * releases, [29] n, [30] end of CTA 0, [31] start. */
#define PAMREC_DEBUG_HEAD_TRACE 2
int pamrec_set_debug(PamrecHandle h, int flags);
int pamrec_head_trace(PamrecHandle h, int backward, uint64_t out[32]);
/* the same run, per CTA: out[barrier * 256 + cta] = %globaltimer (ns) at which CTA `cta` arrived at barrier `barrier` (16 x 256 words) */
int pamrec_head_trace_ctas(PamrecHandle h, int backward, uint64_t* out);

/* Per-launcher device timing: CUDA events recorded on the caller's stream around every launch while enabled.
 * Synchronise the stream, then read (name, accumulated ms, timed launches) per launcher. */
int pamrec_profile_enable(PamrecHandle h, int on);
int pamrec_profile_reset(PamrecHandle h);
int pamrec_profile_count(PamrecHandle h);
int pamrec_profile_get(PamrecHandle h, int index, char name[64], double* total_ms, int64_t* launches);

/* ---- Host input pipeline (no GPU needed).  The batching algorithm of the reference's SequentialIterator over a file that the
 * host has tokenised once into flat columns: io/sequential_iterator.py:475-763 (train branch: per-user history state, listwise
 * groups of 5, round-robin passes, tail batch), :375-474 (eval branch) and :1009-1141 (_convert_data: padding, masks, buckets,
 * satisfied-only compaction).  Output is bit-identical to the reference's 19 feed arrays.  Python's `random` stays with the
 * caller: it passes the shuffled order of the qualifying users and their warm-up lengths (IT:542-545, IT:622). */
typedef struct PamrecBatcher_* PamrecBatcher;
typedef struct PamrecLines {
  int64_t n_lines;
  const int64_t* offsets;       /* [n_lines + 1] into the five history columns (all five have equal length per line)  */
  const int32_t* items; const int32_t* cates;              /* vocabulary indices                                        */
  const double* durs; const double* sats; const double* plays;  /* seconds / 0-1 flags / seconds, as parsed (float64)  */
  const int32_t* user_ids;      /* [n_lines]                                                                           */
  /* eval files (one impression per line); NULL for train files */
  const double* label_sat; const double* label_play; const int32_t* tgt_item; const int32_t* tgt_cate; const double* tgt_dur;
} PamrecLines;
/* the caller keeps the column arrays alive for the batcher's lifetime; borders = decile borders of play / duration (IT:24-42) */
int pamrec_batcher_create(const PamrecLines* lines, const double* borders, int n_borders, int max_seq_len, PamrecBatcher* out);
int pamrec_batcher_destroy(PamrecBatcher b);
/* one training epoch: order[k] = line of the k-th user after random.shuffle, begin_loc[k] = its warm-up length */
int pamrec_batcher_begin_train(PamrecBatcher b, const int64_t* order, const int32_t* begin_loc, int64_t n);
int pamrec_batcher_begin_eval(PamrecBatcher b, int min_seq_length);
/* fills up to batch_size rows of the 19 arrays (order of SequentialIterator.gen_feed_dict, IT:1155-1175; int32 ids, float32
 * values, [rows] or [rows, max_seq_len]); returns the rows written, 0 when the pass is exhausted, < 0 on error */
int pamrec_batcher_next(PamrecBatcher b, int batch_size, void* const* arrays);
/* data parallel: the same GLOBAL batch is drawn, but only the units rank `rank` of `world` trains on / scores are written
 * (listwise groups rank, rank + world, ... of a training batch; rows likewise of an eval batch), compacted to the front of
 * the arrays.  Returns this rank's rows (may be 0 while *global_rows > 0); *global_rows = 0 when the pass is exhausted.
 * Every rank running the same pass with its own rank sees the same sequence of global batches.  global_labels_satisfied /
 * global_users (optional, batch_size floats each) receive those two columns for EVERY row of the global batch: the scoring
 * loops compute their metrics over all rows on every rank (sequential_base_model.py:440-464). */
int pamrec_batcher_next_shard(PamrecBatcher b, int batch_size, int world, int rank, void* const* arrays,
                              float* global_labels_satisfied, float* global_users, int* global_rows);

/* ---- Tokeniser (host only): parser_one_line / parse_file of the reference (io/sequential_iterator.py:195-332) over a whole
 * data file, producing the flat columns of PamrecLines.  `train` selects the 6-column line (one user per line) or the
 * 11-column line (one impression per line).  A vocabulary is the reference's pickled dict given as UTF-8 key bytes:
 * key i = bytes[offsets[i] .. offsets[i+1]), index values[i]; unknown tokens map to 0 (`dict.get(token, 0)`).
 * Returns 0, < 0 on IO / argument errors, or PAMREC_TOK_FALLBACK when the file holds anything outside the strict subset this
 * parser converts bit-identically to Python (non-ASCII bytes, a lone CR, numeric tokens other than plain decimals, ragged or
 * missing columns): the caller then runs the Python parser, which also raises the reference's exceptions for bad lines. */
#define PAMREC_TOK_FALLBACK 1
typedef struct PamrecTokens_* PamrecTokens;
typedef struct PamrecVocab { int64_t n; const char* bytes; const int64_t* offsets; const int32_t* values; } PamrecVocab;
int pamrec_tokenize_file(const char* path, int train, const PamrecVocab* users, const PamrecVocab* items, const PamrecVocab* cates,
                         int n_threads /* 0 = all host cores */, PamrecTokens* out, int64_t* n_lines, int64_t* n_tokens);
/* copies the columns into caller-allocated arrays: dst->n_lines must equal n_lines, offsets has n_lines + 1 entries, the five
 * history columns n_tokens each, the per-line columns n_lines each (the five eval columns are ignored for a train file) */
int pamrec_tokens_read(PamrecTokens t, const PamrecLines* dst);
int pamrec_tokens_free(PamrecTokens t);

/* ---- Checkpoint support (host only): CRC-32C (Castagnoli) as stored, masked, in TensorFlow tensor-bundle checkpoints - the
 * format the reference's tf.train.Saver writes (models/base_model.py:62, :401-417).  `crc` is the value returned for the bytes
 * before `data` (0 to start).  The _portable variant never uses the CPU's crc32 instruction (the two are tested equal). */
uint32_t pamrec_crc32c(uint32_t crc, const void* data, size_t n);
uint32_t pamrec_crc32c_portable(uint32_t crc, const void* data, size_t n);

/* number of kernel launches issued by the last device call on this handle */
int64_t pamrec_last_launch_count(PamrecHandle h);

#ifdef __cplusplus
}
#endif
#endif /* PAMREC_B200_H_ */
