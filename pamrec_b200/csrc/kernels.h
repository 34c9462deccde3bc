// Launcher declarations shared by the translation units of libpamrec_b200.so.
#pragma once
#include <string>
#include <vector>

#include "common.cuh"

namespace pamrec {

// Launch accounting + optional per-launcher device timing (CUDA events on the launching stream).
struct Prof {
  bool on = false;
  int64_t launches = 0;
  std::vector<std::string> names;
  std::vector<double> ms;
  std::vector<int64_t> cnt;
  struct Pair { cudaEvent_t a, b; int id; };
  std::vector<Pair> pending;
  std::vector<cudaEvent_t> free_ev;
  int id_of(const char* name);
  cudaEvent_t get_event();
  void resolve();          // caller has synchronised the stream
  void reset();
  ~Prof();
};
extern thread_local Prof* g_prof;
struct ProfScope {
  Prof* p; cudaStream_t st; cudaEvent_t b; bool timed;
  ProfScope(const char* name, int n_kernels, cudaStream_t st);
  ~ProfScope();
};
#define PAMREC_PROF(name, n, st) ProfScope _prof_scope(name, n, st)

// ---- kernels_encoder.cu
int init_encoder_kernels(int max_T);   // per-device opt-in to > 48 KB dynamic shared memory (called by pamrec_bind)
void launch_embed_fwd(const int* ih, const int* ch, const int* items, const int* cates, const float* item_w,
                      const float* cate_w, const float* pos, float* x0, float* tgt, int64_t n_rows, int T, cudaStream_t st);
void launch_bucket_plan(const float* lt, int n, int* bucket, int* perm, int* ctl, int* tile_bucket, int* tile_begin,
                        int* tile_count, cudaStream_t st);
void launch_proj_fwd(const float* X, const int* perm, const int* ctl, const int* tile_bucket, const int* tile_begin,
                     const int* tile_count, int max_tiles, const float* Wq, const float* Wk, const float* Wv,
                     const float* ln_beta, const float* ln_gamma, float* QIN, float* Q, float* K, float* V, cudaStream_t st);
void launch_attn_fwd(const float* Q, const float* K, const float* V, const float* QIN, const int* mask, float* Y, float* PV,
                     float* ML, int B, int T, cudaStream_t st);
void launch_ffn_fwd(const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                    const float* ln_beta, const float* ln_gamma, float* OUT, float* Hdbg, int n_tok, cudaStream_t st);
// dOUT_keep (nullable): receives a copy of dOUT for launch_enc_dw, when the buffer dOUT is overwritten before that runs
void launch_ffn_bwd(const float* Y, const float* dOUT, const float* W1, const float* b1, const float* W2,
                    const float* ln_beta, const float* ln_gamma, float* dY, float* H, float* DHR, float* dOUT_keep,
                    float* dbeta, float* dgamma, int n_tok, cudaStream_t st);
void launch_attn_bwd(const float* Q, const float* K, const float* V, const float* dY, const float* PV, const float* ML,
                     const int* mask, float* dQ, float* dK, float* dV, int B, int T, cudaStream_t st);
void launch_proj_bwd(const float* X, const float* dY, const float* dQ, const float* dK, const float* dV, const int* perm,
                     const int* ctl, const int* tile_bucket, const int* tile_begin, const int* tile_count, int max_tiles,
                     const float* Wq, const float* Wk, const float* Wv, const float* ln_beta, const float* ln_gamma,
                     float* dX, float* dbeta, float* dgamma, cudaStream_t st);
// weight gradients of one encoder block from what its backward pass saved (kernels_encoder.cu:k_enc_dw); accumulated atomically
struct EncDwArgs {
  const float* qin; const float* x; const float* dQ; const float* dK; const float* dV;   // projection: [N, 40] each
  const int* perm; const int* ctl;                                                       // bucket sort (launch_bucket_plan)
  const float* y; const float* ln_beta; const float* ln_gamma;                           // f = LN_b(y)
  const float* h; const float* dhr; const float* dout;                                   // relu(f W1 + b1), dH o relu', dOUT
  float* dWq; float* dWk; float* dWv;                                                    // [10, 40, 40]
  float* dW1; float* db1; float* dW2; float* db2;
  int n_tok;
  bool ffn;                                                                              // the FFN pair, else the projection
};
void launch_enc_dw(const EncDwArgs& a, cudaStream_t st);

// ---- kernels_attn_mma.cu (attention forward + backward on warp-level tensor-core MMAs, 3xTF32; used up to T = 128)
int init_attn_mma_kernels(int max_T);
void launch_attn_fwd_mma(const float* Q, const float* K, const float* V, const float* QIN, const int* mask, float* Y, float* PV, float* ML,
                         int B, int T, cudaStream_t st);
void launch_attn_bwd_mma(const float* Q, const float* K, const float* V, const float* dY, const float* PV, const float* ML,
                         const int* mask, float* dQ, float* dK, float* dV, int B, int T, cudaStream_t st);

// ---- kernels_head.cu
void launch_dense_fwd(const DenseP& p, cudaStream_t st);
void launch_dense_dx(const DenseDxP& p, cudaStream_t st);
void launch_dense_dw(const DenseDwP& p, cudaStream_t st);
void launch_bn_finalize(const BnSet& s, double count, cudaStream_t st);   // training: sums -> stat, moving update, sums := 0
void launch_bn_eval_stat(const BnSet& s, cudaStream_t st);                // inference: stat from moving stats
void launch_bn_bwd_stats(const BnSet& s, const float* dA, const float* Z, int M, cudaStream_t st);
void launch_pool_fwd(const float* H, const float* Z2, const BnSet& s1, const int* mask, float* new_long, int B, int T,
                     cudaStream_t st);
void launch_pool_bwd(const float* H, const float* Z2, const BnSet& s1, const int* mask, const float* d_new_long, float* dA2,
                     float* dH, int B, int T, cudaStream_t st);
void launch_combine_fwd(const float* ZE1, const float* ZG1, const BnSet& e1, const BnSet& g1, const float* tgt, float* U,
                        int B, cudaStream_t st);
void launch_combine_bwd(const float* ZE1, const float* ZG1, const BnSet& e1, const BnSet& g1, const float* dU, float* dE1,
                        float* dG1, float* dTgt, int B, cudaStream_t st);
// loss_acc (double[8]): [0] data [1] aux [2] order (all already weighted / averaged)
void launch_loss(const float* logits, const float* y_sat, const float* y_play, const float* plays, float* d_logits,
                 double* loss_acc, int B, int B_global, const double* n_valid_global, float fuzhu_w, float order_w,
                 int softmax_group, cudaStream_t st);   // softmax_group = 0: sigmoid cross entropy heads
void launch_sigmoid_col0(const float* logits, float* pred, int B, cudaStream_t st);

// ---- kernels_optim.cu
struct SparseTable {
  int width;                  // floats per row: 4, 8, 16, 20, 32 or 40 (the sparse kernels refuse any other width)
  int64_t n_rows;
  float* w; float* m; float* v;
  int* keys; int* idx; int* skeys; int* sidx; int* uidx; int* ukeys; int* slot;
  float* accum;               // [n_keys, width]
  int* nuniq;                 // device scalar
  double* normsq;             // device scalar: sum of squares of every un-deduplicated gradient row
  const int* l2_has0;         // nullable device flag; when it reads 0, row 0 is looked up but carries no L2 term (sibling models: the
                              // padding id of the satisfied-only history, kernels_sibling.cu:k_sib_has0)
};
// undedup (nullable): [0] += sum of squares of every item gradient row (history and target lookups), [1] likewise category rows
void launch_embed_bwd_reduce(const float* dX0, const float* dTgtHead, float* dTgtTotal, float* dPos, double* pos_normsq,
                             double* undedup, int B, int T, cudaStream_t st);
size_t sparse_temp_bytes(int64_t n_keys);
// builds keys (history ids then target ids), sorts, finds unique rows, reduces duplicate rows into accum
int launch_sparse_reduce(const SparseTable& t, const int* hist_ids, const int* tgt_ids, int64_t n_hist, int64_t n_tgt,
                         const float* hist_grad, int hist_ld, int hist_col, const float* tgt_grad, int tgt_ld, int tgt_col,
                         void* cub_temp, size_t cub_bytes, cudaStream_t st);
int launch_sparse_plan(const SparseTable& t, const int* hist_ids, const int* tgt_ids, int64_t n_hist, int64_t n_tgt,
                       int world, int64_t rps, int64_t key_range, bool fill_slot, void* cub_temp, size_t cub_bytes,
                       cudaStream_t st);
// launch_sparse_segreduce / _l2norm / _adam return -1 (nothing launched) for a table width they have no instantiation for
int launch_sparse_segreduce(const SparseTable& t, int64_t n, int64_t n_hist, const float* hist_grad, int hist_ld, int hist_col,
                            const float* tgt_grad, int tgt_ld, int tgt_col, double* normsq, cudaStream_t st);
void launch_slot_reset(const SparseTable& t, int64_t n_keys, cudaStream_t st);
// L2 rows of the unique ids: adds their squared norm to normsq and 0.5*l2*|w|^2 to reg_acc
int launch_sparse_l2norm(const SparseTable& t, int64_t n_keys, float l2, double* reg_acc, cudaStream_t st);
int launch_sparse_adam(const SparseTable& t, int64_t n_keys, int mode, float l2, float lr_t, float b1, float b2, float eps,
                        float clip, int is_clip, cudaStream_t st);
void launch_dense_norm(const float* P, const float* G, const int* seg_tab, int n_seg, float layer_l2, double* seg_normsq,
                       const double* pos_normsq, double* reg_acc, cudaStream_t st);
void launch_dense_adam(float* P, const float* G, float* M, float* V, const int* seg_id, const int* seg_tab,
                       const double* seg_normsq, int64_t n, float layer_l2, float lr_t, const float* lr_dev, float b1, float b2, float eps,
                       float clip, int is_clip, cudaStream_t st);
// step > 0: *step_dev = step; step == 0: *step_dev += 1 (graph replay).  *lr_out = lr * sqrt(1 - b2^t) / (1 - b1^t) in double, as
// the host computes it (base_model.py:270-271 + TF 2.4 AdamOptimizer._prepare)
void launch_adam_step(int64_t step, double* step_dev, float lr, float b1, float b2, float* lr_out, cudaStream_t st);
// l2sq (nullable): |w|^2 of the unique looked-up rows per table (kernels_sparse2.cu) - their share of the regularisation loss
// and of the clip norms (added to sp_normsq[0..3] here, after every consumer has run, so that sp_normsq reads as the full norm)
void launch_finish_losses(const double* loss_acc, float* losses, const double* l2sq, float embed_l2, double* sp_normsq, cudaStream_t st);

// ---- kernels_sparse2.cu (one-sort plan, run walk with fused Adam; local and replicated tables)
enum { SP2_COMPACT = 0,   // DENSE_EXACT on local tables: run sums -> compact accumulator, row -> unique index map, full sweep
       SP2_FUSED = 1,     // LAZY on local tables: Adam applied to the row inside the walk
       SP2_DENSE = 2 };   // replicated tables (data parallel): run sums -> dense gradient table + touch counts, all-reduced, sweep
// lr = lr_t of TF's Adam (learning rate with both bias corrections); lr_dev != null: read it from device memory instead (the
// step counter lives on the device when the step is replayed from a CUDA graph, kernels_optim.cu:k_adam_step)
struct AdamP { float lr, b1, b2, eps, l2, clip; int is_clip; const float* lr_dev; };
struct Sp2 {
  const int* item_hist; const int* cate_hist; const int* items; const int* cates; const int* users;
  int64_t N; int B;                                  // history positions (B * T), rows
  int n_items, n_cates, n_users;
  int* keys; int* idx; int* skeys; int* sidx; int* uidx;   // [2 (N + B) + B]: item lookups | category lookups | users
  int* ukeys[3]; int* nuniq;                         // per table: sorted unique ids, their count (nuniq[0..2])
  int* meta;                                         // [0..2] global unique index of the first run of table t, [3] total
  int* slot;                                         // COMPACT: [n_items + n_cates + n_users] row -> unique index of its table, or -1
  float* accum[2]; int* dflag[2];                    // compact run sums [unique][width]; FUSED: rows left to k_sp2_lazy_finish
  double* l2sq;                                      // [4] item cate user_long user_short: |w|^2 over the unique rows
  const double* undedup;                             // [4] squared norm of the un-deduplicated gradient rows (sp_normsq)
  float* w[4]; float* m[4]; float* v[4];             // item cate user_long user_short
  const float* dX0; const float* dT;                 // [N,40] token gradients (item 0:16, cate 16:20); [B,20] target-row gradients
  float* rep_grad;                                   // DENSE: G_item [n_items,16] | G_cate [n_cates,4] | touch [n_items+n_cates+n_users]
  int mode;
};
inline int64_t sp2_rep_floats(int64_t n_items, int64_t n_cates, int64_t n_users) { return n_items * 17 + n_cates * 5 + n_users; }
size_t sp2_temp_bytes(int64_t n_keys);
int launch_sp2_plan(const Sp2& s, void* cub_temp, size_t cub_bytes, cudaStream_t st);
void launch_sp2_walk(const Sp2& s, const AdamP& a, cudaStream_t st);
void launch_sp2_lazy_finish(const Sp2& s, const AdamP& a, cudaStream_t st);
void launch_sp2_adam_sweep(const Sp2& s, const AdamP& a, int lazy, cudaStream_t st);
void launch_sp2_rep_l2(const Sp2& s, cudaStream_t st);

// ---- kernels_sibling.cu (MMoE_original / PLE / ShareBottom: DIN attention pooling, mixing, loss); item_dim = 16 or 32 (cate = item / 4)
void launch_sib_gather(const int* sat_item, const int* sat_cate, const int* hist_item, const int* hist_cate, const int* items,
                       const int* cates, const float* item_w, const float* cate_w, float* h, float* tgt, int* ids_item,
                       int* ids_cate, int B, int T, int item_dim, cudaStream_t st);
void launch_sib_has0(const int* hist_item, const int* hist_cate, const int* items, const int* cates, int B, int T, int* has0,
                     cudaStream_t st);
void launch_sib_feat_fwd(float* feat, const float* tgt, int B, int T, int item_dim, cudaStream_t st);
void launch_sib_feat_bwd(const float* d_feat, const float* feat, const float* tgt, float* d_att, float* dq, int B, int T, int item_dim,
                         cudaStream_t st);
void launch_sib_pool_fwd(const float* h, const float* score, const int* sat_mask, const int* mask, const float* tgt, float* aw,
                         float* x, int B, int T, int item_dim, cudaStream_t st);
void launch_sib_pool_bwd(const float* h, const float* aw, const int* sat_mask, const int* mask, const float* d_x, float* d_score,
                         float* dh, int B, int T, int item_dim, cudaStream_t st);
void launch_sib_tgt_total(const float* d_tgt, const float* d_x, const float* dq, float* out, int B, int item_dim, cudaStream_t st);
void launch_sib_mix_fwd(const float* ZE1, const float* ZG1, const BnSet& e1, const BnSet& g1, const float* tgt, float* U, int n_expert,
                        const int sel[2][5], int B, int item_dim, cudaStream_t st);
void launch_sib_mix_bwd(const float* ZE1, const float* ZG1, const BnSet& e1, const BnSet& g1, const float* dU, float* dE1, float* dG1,
                        float* dTgt, int n_expert, const int sel[2][5], int B, int item_dim, cudaStream_t st);
// heads = 2: logits [B,2] (satisfied label, play label x aux_w); heads = 1: logits [B,1], data loss only (SASRec)
void launch_sib_loss(const float* logits, const float* y_sat, const float* y_play, float* d_logits, double* loss_acc, int B, float aux_w,
                     int heads, cudaStream_t st);
void launch_sib_pred(const float* logits, float* pred, int B, int heads, cudaStream_t st);

// ---- kernels_sasrec.cu (SASRecModel: two S-wide self-attention blocks with dense Q / K / V; S = item + cate width, 20 or 40)
int init_sas_kernels(int max_T);       // opt-in to > 48 KB dynamic shared memory of the S = 40 attention kernels (called by pamrec_bind)
void launch_sas_embed(const float* h, const float* pos, float* x0, int B, int T, int S, cudaStream_t st);
void launch_sas_proj_fwd(const float* X, const float* W, const float* bias, const float* ln_beta, const float* ln_gamma, float* XQ,
                         float* QKV, int64_t N, int S, cudaStream_t st);
void launch_sas_proj_bwd(const float* XQ, const float* dQKV, const float* dY, const float* W, const float* ln_gamma, float* dX,
                         float* g_gamma, float* g_beta, int64_t N, int S, cudaStream_t st);
void launch_sas_attn_fwd(const float* QKV, const float* XQ, const int* mask, float* Y, float* ML, int B, int T, int S, cudaStream_t st);
void launch_sas_attn_bwd(const float* QKV, const float* XQ, const float* Y, const float* dY, const float* ML, const int* mask, float* dQKV,
                         float* Dq, int B, int T, int S, cudaStream_t st);
void launch_sas_ffn_fwd(const float* Y, const float* W1, const float* b1, const float* W2, const float* b2, const float* ln_beta,
                        const float* ln_gamma, float* F, float* HPRE, float* OUT, int64_t N, int S, cudaStream_t st);
void launch_sas_ffn_bwd(const float* Y, const float* HPRE, const float* dOUT, const float* W1, const float* W2, const float* ln_gamma,
                        float* HID, float* DHPRE, float* dY, float* g_gamma, float* g_beta, int64_t N, int S, cudaStream_t st);
void launch_sas_final_fwd(const float* SEQ, const int* mask, const float* tgt, float* U, int B, int T, int S, cudaStream_t st);
void launch_sas_final_bwd(const float* dU, const int* mask, float* dSEQ, float* dTgt, int B, int T, int S, cudaStream_t st);
void launch_sas_pos_bwd(const float* dX0, float* dPos, double* normsq, int B, int T, int S, cudaStream_t st);

// ---- kernels_p2p.cu + kernels_head2.cu (data-parallel exchanges through NVLink peer mailboxes)
constexpr int kP2PMaxDoubles = 2048;     // payload capacity of one mailbox slot (expert + gate layer-0 sums: 1256)
constexpr int kP2PSlots = 24;            // sync points per step (each has its own slot): 12 forward + 12 backward barriers
constexpr int kP2PMaxWorld = 8;
// A mailbox starts with a 256-byte header whose first word is the rank's error word (0 = ok; a peer that never arrived: 1 + slot from
// the persistent head kernels, 200 + flag set from k_xr_*).  Then the flag-in-data region of the persistent head kernels: 16 bytes
// per double ({low word, epoch, high word, epoch}: the arrival of the data IS the signal - one NVLink trip per exchange instead of
// payload, system fence, flag)
constexpr size_t p2p_ll_offset() { return 256; }
// ... then the gradient exchange region of k_xr_* (kernels_p2p.cu): flags | scalars | own contribution | reduced result
constexpr int kXrScalars = 16;           // doubles per rank travelling with the gradients (8 clip norms + 4 loss sums)
inline size_t p2p_xr_offset(int world) { return (p2p_ll_offset() + (size_t)kP2PSlots * world * kP2PMaxDoubles * 16 + 255) / 256 * 256; }
inline int64_t p2p_xr_cap(int world, int64_t n_floats) { const int64_t q = 64 * (int64_t)world; return (n_floats + q - 1) / q * q; }
inline size_t p2p_xr_header_bytes() { return 512 + (size_t)kP2PMaxWorld * kXrScalars * sizeof(double); }
inline size_t p2p_mailbox_bytes(int world, int64_t xr_floats) {
  return p2p_xr_offset(world) + p2p_xr_header_bytes() + 2 * (size_t)p2p_xr_cap(world, xr_floats) * sizeof(float);
}
// All-reduce (sum) of the gradient buffers of a data-parallel step through peer memory, two-shot: every rank sums ITS slice of all
// ranks' contributions (reads over NVLink, rank order) and writes the result into every rank's result buffer.
struct XrArgs {
  char* peer[kP2PMaxWorld];               // every rank's exchange region (own one included)
  int world, rank; uint32_t epoch;
  int64_t cap;                            // floats of one contribution (multiple of 64 * world)
  const float* dense_grad; int64_t n_dense;   // packed into the front of the contribution; the reduced values are copied back
  double* scalars[2]; int n_scalars[2];   // fp64 scalars reduced alongside (in place)
  unsigned* counter;                      // device words for the "last CTA" hand-off (3 words)
  uint32_t* err;
};
inline float* xr_xbuf(char* region) { return reinterpret_cast<float*>(region + p2p_xr_header_bytes()); }
void launch_xr_allreduce(const XrArgs& a, float* dense_grad_out, cudaStream_t st);

// ---- kernels_shard.cu (row-sharded tables)
void launch_shard_route(const SparseTable& req, int64_t n, int world, int64_t rps, int* off, int* counts, int slot, int* send_ids,
                        int* inv, cudaStream_t st);
void launch_serve_rows(const float* shard, const int* ids, int64_t n, int width, float* out, cudaStream_t st);
void launch_count_valid_groups(const float* plays, int B, double* out, cudaStream_t st);

}  // namespace pamrec
