// Host-side description of the model: where every TF variable (SURVEY.md Appendix B) lives in
// the caller's flat pools, and how the workspace is carved.  No CUDA calls in here, so the
// inventory can be queried on a machine without a GPU.
#pragma once
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "common.cuh"

namespace pamrec {

struct TensorDesc {
  std::string name;
  int pool = 0, dtype = PAMREC_F32, flags = 0;
  int64_t offset = 0, numel = 0;
  int ndim = 0;
  int64_t shape[4] = {0, 0, 0, 0};
};

struct BlockOff { int64_t ln_a_beta, ln_a_gamma, wq, wk, wv, w1, b1, w2, b2, ln_b_beta, ln_b_gamma; };
// 2-layer BN MLP, group-strided: offset of group 0; group g lives at off + g * (numel of one member)
struct MlpOff { int64_t w0, b0, g0, be0, w1, b1, g1, be1, wout, bout; };
struct BnOff { int C; int64_t gamma, beta, mm, mv; };

enum BnId { BN_S0 = 0, BN_S1, BN_E0, BN_G0, BN_E1, BN_G1, BN_T0, BN_T1, BN_COUNT };

// one row-sharded table as seen by the exchange (PAMREC_TABLES_SHARDED)
struct ShardDim { int64_t vocab = 0, rps = 0, nk = 0, cap_recv = 0; int width = 0; };

struct Layout {
  int n_users = 0, n_items = 0, n_cates = 0, T = 0, Bcap = 0;
  int world = 1, table_mode = 0;
  ShardDim sh_item, sh_cate, sh_user;
  int64_t cub_keys = 0;                         // largest key count handed to cub
  int64_t cub_keys_table = 0;                   // lookups of one table per batch (N + B)
  int64_t rows_of(int64_t vocab) const { return table_mode == PAMREC_TABLES_SHARDED ? (vocab + world - 1) / world : vocab; }
  std::vector<TensorDesc> dense, bn, ws;
  int64_t dense_numel = 0, bn_numel = 0;
  size_t ws_bytes = 0;
  int64_t pos = 0;
  BlockOff blk[2];
  MlpOff score, expert, gate, tower;
  BnOff bnoff[BN_COUNT];
  int64_t bn_bsums_off[BN_COUNT];
  std::map<std::string, size_t> ws_index;
  // sibling models (PAMREC_MODEL_MMOE / _PLE / _SHAREBOTTOM, build_sibling below): the attention MLP of the two DIN branches
  // takes the place of the score MLP (BN_S0 / BN_S1 = its two layers, 2 x 80 and 2 x 40 channels)
  int model_kind = PAMREC_MODEL_PAMREC;
  int n_expert = 0;                             // 5 (MMoE), 7 (PLE: 3 shared, 2 main, 2 sub), 0 (share-bottom)
  int gate_sel[2][5] = {{0, 1, 2, 3, 4}, {0, 1, 2, 3, 4}};   // experts mixed by gate_main / gate_sub (ple.py:51-58)
  int tower_in = 0;                             // 64 + E (mixing output | target) or 3 E (share-bottom: x itself)
  MlpOff att;                                   // att_fcn of long_term, short_term (group-strided)
  int64_t att_mat = 0;                          // attention_mat of long_term; short_term follows at + emb_dim^2
  // embedding widths (pamrec_create has validated them): item | cate = one history token of emb_dim floats; PAMRec: 16 / 4 / 20
  int item_dim = kI, cate_dim = kC, user_dim = PAMREC_USER_DIM, emb_dim = kE;

  int64_t add_dense(const std::string& name, std::initializer_list<int64_t> shape, int flags) {
    TensorDesc t;
    t.name = name; t.pool = PAMREC_POOL_DENSE; t.flags = flags; t.offset = dense_numel;
    t.numel = 1; t.ndim = 0;
    for (int64_t s : shape) { t.shape[t.ndim++] = s; t.numel *= s; }
    dense_numel += t.numel;
    dense.push_back(t);
    return t.offset;
  }
  int64_t add_bn(const std::string& name, int64_t n) {
    TensorDesc t;
    t.name = name; t.pool = PAMREC_POOL_BN; t.offset = bn_numel; t.numel = n; t.ndim = 1; t.shape[0] = n;
    bn_numel += n;
    bn.push_back(t);
    return t.offset;
  }
  void add_ws(const std::string& name, int dtype, std::initializer_list<int64_t> shape) {
    TensorDesc t;
    t.name = name; t.pool = PAMREC_POOL_WORKSPACE; t.dtype = dtype; t.offset = (int64_t)ws_bytes;
    t.numel = 1; t.ndim = 0;
    for (int64_t s : shape) { t.shape[t.ndim++] = s; t.numel *= s; }
    size_t esz = (dtype == PAMREC_F64) ? 8 : (dtype == PAMREC_U8 ? 1 : 4);
    size_t bytes = (size_t)t.numel * esz;
    ws_bytes += (bytes + 255) / 256 * 256;
    ws_index[name] = ws.size();
    ws.push_back(t);
  }
  size_t ws_off(const std::string& name) const {
    auto it = ws_index.find(name);
    if (it == ws_index.end()) { fprintf(stderr, "pamrec: unknown workspace tensor %s\n", name.c_str()); abort(); }
    return (size_t)ws[it->second].offset;
  }

  // members: TF scope of each group member; sizes in->h0->h1(->1)
  MlpOff add_mlp(const std::vector<std::string>& scopes, const std::vector<int>& flags, int in, int h0, int h1, bool out,
                 BnOff* bn0, BnOff* bn1, bool live = true) {
    MlpOff o{};
    auto role = [&](const char* leaf, std::initializer_list<int64_t> shape) {
      int64_t first = -1;
      for (size_t g = 0; g < scopes.size(); ++g) {
        int64_t off = add_dense(scopes[g] + "/nn_part/" + leaf, shape, flags[g]);
        if (g == 0) first = off;
      }
      return first;
    };
    o.w0 = role("w_nn_layer0", {in, h0});
    o.b0 = role("b_nn_layer0", {h0});
    o.g0 = role("batch_normalization/gamma", {h0});
    o.be0 = role("batch_normalization/beta", {h0});
    o.w1 = role("w_nn_layer1", {h0, h1});
    o.b1 = role("b_nn_layer1", {h1});
    o.g1 = role("batch_normalization_1/gamma", {h1});
    o.be1 = role("batch_normalization_1/beta", {h1});
    o.wout = o.bout = -1;
    if (out) {
      o.wout = role("w_nn_output", {h1, 1});
      o.bout = role("b_nn_output", {1});
    }
    int G = (int)scopes.size();
    int64_t mm0 = -1, mv0 = -1, mm1 = -1, mv1 = -1;
    for (int g = 0; g < G; ++g) { int64_t x = add_bn(scopes[g] + "/nn_part/batch_normalization/moving_mean", h0); if (!g) mm0 = x; }
    for (int g = 0; g < G; ++g) { int64_t x = add_bn(scopes[g] + "/nn_part/batch_normalization/moving_variance", h0); if (!g) mv0 = x; }
    for (int g = 0; g < G; ++g) { int64_t x = add_bn(scopes[g] + "/nn_part/batch_normalization_1/moving_mean", h1); if (!g) mm1 = x; }
    for (int g = 0; g < G; ++g) { int64_t x = add_bn(scopes[g] + "/nn_part/batch_normalization_1/moving_variance", h1); if (!g) mv1 = x; }
    if (bn0) *bn0 = BnOff{G * h0, o.g0, o.be0, mm0, mv0};
    if (bn1) *bn1 = BnOff{G * h1, o.g1, o.be1, mm1, mv1};
    (void)live;
    return o;
  }

  // optimiser scratch shared by every model family
  void add_optim_ws() {
    add_ws("seg_id", PAMREC_I32, {dense_numel});
    add_ws("seg_tab", PAMREC_I32, {(int64_t)dense.size(), 4});   // off, numel, flags, -
    add_ws("seg_normsq", PAMREC_F64, {(int64_t)dense.size()});
    add_ws("sp_normsq", PAMREC_F64, {8});          // 0 item 1 cate 2 ulong 3 ushort 4 pos
    add_ws("adam.step", PAMREC_F64, {2});          // optimiser step on the device (graph replay advances it there)
    add_ws("adam.lr", PAMREC_F32, {4});            // lr_t of the current step, written by k_adam_step
  }
  void add_bn_ws() {
    const char* bn_names[BN_COUNT] = {"s0", "s1", "e0", "g0", "e1", "g1", "t0", "t1"};
    int64_t bn_c = 0;
    for (int i = 0; i < BN_COUNT; ++i) {
      std::string p = std::string("bn.") + bn_names[i];
      add_ws(p + ".sums", PAMREC_F64, {bnoff[i].C, 2});
      add_ws(p + ".stat", PAMREC_F32, {bnoff[i].C, 2});
      bn_bsums_off[i] = 2 * bn_c;
      bn_c += bnoff[i].C;
    }
    add_ws("bn.bsums", PAMREC_F64, {bn_c, 2});   // backward sums (sum dy, sum dy*xhat) of all sets: one memset per step
    add_ws("bn.gsums", PAMREC_F64, {8, bn_c, 2});    // row-stationary head: 8 copies of the forward sums (set-major inside a copy group)
    add_ws("bn.gbsums", PAMREC_F64, {8, bn_c, 2});   // ... and of the backward sums
  }

  // MMoEModel_original / PLEModel / ShareBottomModel (oracle/siblings_oracle.py:param_spec has the same inventory, by TF name)
  void build_sibling(const PamrecConfig& c) {
    const int L2 = PAMREC_SEG_L2;
    const int64_t B = Bcap, N = (int64_t)Bcap * T;
    const int E = emb_dim;
    const std::string clsr = "sequential/clsr/";
    // ---- dense pool
    att_mat = add_dense(clsr + "long_term/attention_fcn/attention_mat", {E, E}, L2);          // mmoe.py:315-319
    add_dense(clsr + "short_term/attention_fcn/attention_mat", {E, E}, L2);
    att = add_mlp({clsr + "long_term/attention_fcn/att_fcn", clsr + "short_term/attention_fcn/att_fcn"}, {L2, L2}, 4 * E, 80, 40, true,
                  &bnoff[BN_S0], &bnoff[BN_S1]);                                                 // mmoe.py:327-329
    const int x_dim = 3 * E;
    std::vector<std::string> ex;
    if (model_kind == PAMREC_MODEL_MMOE) {
      for (int j = 0; j < 5; ++j) ex.push_back(clsr + "expert_" + std::to_string(j));           // mmoe.py:38-41
    } else if (model_kind == PAMREC_MODEL_PLE) {
      for (int j = 0; j < 3; ++j) ex.push_back(clsr + "share_expert_" + std::to_string(j));     // ple.py:38-49
      for (int j = 0; j < 2; ++j) ex.push_back(clsr + "main_expert_" + std::to_string(j));
      for (int j = 0; j < 2; ++j) ex.push_back(clsr + "sub_expert_" + std::to_string(j));
      const int ms[5] = {0, 1, 2, 3, 4}, ss[5] = {0, 1, 2, 5, 6};                              // shared experts first (ple.py:51-58)
      for (int j = 0; j < 5; ++j) { gate_sel[0][j] = ms[j]; gate_sel[1][j] = ss[j]; }
    }
    n_expert = (int)ex.size();
    if (n_expert) {
      expert = add_mlp(ex, std::vector<int>(ex.size(), L2), x_dim, 100, 64, false, &bnoff[BN_E0], &bnoff[BN_E1]);
      gate = add_mlp({clsr + "gate_main", clsr + "gate_sub"}, {L2, L2}, x_dim, 64, 5, false, &bnoff[BN_G0], &bnoff[BN_G1]);
      tower_in = 64 + E;
    } else {
      bnoff[BN_E0] = bnoff[BN_E1] = bnoff[BN_G0] = bnoff[BN_G1] = BnOff{0, 0, 0, 0, 0};
      tower_in = x_dim;                                                                          // sharebottom.py:200-201
    }
    tower = add_mlp({"sequential/logit_fcn", "sequential/valid_logit_fcn"}, {L2, L2}, tower_in, 100, 64, true, &bnoff[BN_T0], &bnoff[BN_T1]);
    // ---- workspace.  Branch 0 = long_term (satisfied-only history), branch 1 = short_term (full history).
    add_ws("sib.ids_item", PAMREC_I32, {2, N});      // lookups of the item table in branch order (keys of the sparse plan)
    add_ws("sib.ids_cate", PAMREC_I32, {2, N});
    add_ws("sib.h", PAMREC_F32, {2, N, E});         // gathered history tokens item | cate
    add_ws("tgt", PAMREC_F32, {B, E});
    add_ws("sib.feat", PAMREC_F32, {N, 8 * E});      // per branch: a = h A | q | a - q | a * q   (mmoe.py:320-326)
    add_ws("z1", PAMREC_F32, {N, 160});              // att_fcn layer 0 pre-activations (both branches)
    add_ws("z2", PAMREC_F32, {N, 80});               // layer 1
    add_ws("sib.score", PAMREC_F32, {N, 2});         // linear output = attention logits
    add_ws("sib.aw", PAMREC_F32, {2, N});            // softmax weights, kept for the backward pass
    add_ws("x", PAMREC_F32, {B, x_dim});             // long | short | target
    add_ws("ze0", PAMREC_F32, {B, (int64_t)n_expert * 100});
    add_ws("zg0", PAMREC_F32, {B, n_expert ? 128 : 0});
    add_ws("ze1", PAMREC_F32, {B, (int64_t)n_expert * 64});
    add_ws("zg1", PAMREC_F32, {B, n_expert ? 10 : 0});
    add_ws("u", PAMREC_F32, {B, 2 * (64 + E)});   // main | target | sub | target
    add_ws("zt0", PAMREC_F32, {B, 200});
    add_ws("zt1", PAMREC_F32, {B, 128});
    add_ws("logits", PAMREC_F32, {B, 2});            // logit_fcn (satisfied label), valid_logit_fcn (play label)
    add_ws("losses", PAMREC_F32, {8});
    add_ws("loss_acc", PAMREC_F64, {8});
    add_ws("d_logits", PAMREC_F32, {B, 2});
    add_ws("d_t1", PAMREC_F32, {B, 128});
    add_ws("d_t0", PAMREC_F32, {B, 200});
    add_ws("d_u", PAMREC_F32, {B, 2 * (64 + E)});
    add_ws("d_e1", PAMREC_F32, {B, (int64_t)n_expert * 64});
    add_ws("d_g1", PAMREC_F32, {B, n_expert ? 10 : 0});
    add_ws("d_e0", PAMREC_F32, {B, (int64_t)n_expert * 100});
    add_ws("d_g0", PAMREC_F32, {B, n_expert ? 128 : 0});
    add_ws("d_x", PAMREC_F32, {B, x_dim});
    add_ws("d_tgt", PAMREC_F32, {B, E});            // from the towers' target columns
    add_ws("d_tgt_total", PAMREC_F32, {B, E});
    add_ws("sib.d_score", PAMREC_F32, {N, 2});
    add_ws("sib.d_a1", PAMREC_F32, {N, 80});
    add_ws("sib.d_a0", PAMREC_F32, {N, 160});
    add_ws("sib.d_feat", PAMREC_F32, {N, 8 * E});
    add_ws("sib.d_att", PAMREC_F32, {2, N, E});     // gradient of a = h A
    add_ws("sib.dq", PAMREC_F32, {B, 2, E});        // gradient of the query (target) through the feature rows, per branch
    add_ws("sib.dh", PAMREC_F32, {2, N, E});        // gradient of the gathered tokens = rows of the sparse gradient
    add_ws("sib.zero", PAMREC_F32, {256});           // never written: the bias of the bias-free attention_mat product
    add_ws("sib.dummy", PAMREC_F32, {256});          // sink of that product's bias gradient
    add_ws("sib.has0", PAMREC_I32, {4});             // [0] item [1] category: id 0 occurs among the history / target ids; when it
                                                     // does not, row 0 is looked up by the satisfied-only history's padding alone and
                                                     // is not among the L2 rows (sequential_base_model.py:640-664)
    add_bn_ws();
    add_optim_ws();
    // sparse path (kernels_optim.cu, one plan per table): keys = satisfied ids, history ids, target ids
    const int64_t NK = 2 * N + B;
    cub_keys_table = NK;
    for (const char* t : {"item", "cate"}) {
      std::string p = std::string("sp.") + t + ".";
      for (const char* n : {"keys", "idx", "skeys", "sidx", "uidx", "ukeys"}) add_ws(p + n, PAMREC_I32, {NK});
      add_ws(p + "slot", PAMREC_I32, {t[0] == 'i' ? n_items : n_cates});
      add_ws(p + "accum", PAMREC_F32, {NK, t[0] == 'i' ? item_dim : cate_dim});
    }
    for (const char* n : {"keys", "idx", "skeys", "sidx", "uidx", "ukeys"}) add_ws(std::string("sp.user.") + n, PAMREC_I32, {B});
    add_ws("sp.user.slot", PAMREC_I32, {n_users});
    add_ws("sp.nuniq", PAMREC_I32, {8});
    add_ws("dp.scalars", PAMREC_F64, {8});
    cub_keys = NK;
    add_ws("cub_temp", PAMREC_U8, {(int64_t)(16u << 20) + 16 * cub_keys});
    (void)c;
  }

  // SASRecModel (oracle/siblings_oracle.py:sasrec_param_spec has the same inventory, by TF name)
  struct SasBlock { int64_t ln_a_beta, ln_a_gamma, wqkv, bqkv, ln_b_beta, ln_b_gamma, w1, b1, w2, b2; };
  SasBlock sas[2];
  void build_sasrec(const PamrecConfig& c) {
    const int L2 = PAMREC_SEG_L2;
    const int64_t B = Bcap, N = (int64_t)Bcap * T;
    const int E = emb_dim;
    pos = add_dense("sequential/embedding/position_embedding", {T, E}, PAMREC_SEG_POS);       // sasrec.py:29-34
    for (int b = 0; b < 2; ++b) {
      const std::string p = "sequential/sasrec/num_blocks_" + std::to_string(b) + "/";
      SasBlock& o = sas[b];
      // Q, K, V kernels adjacent (one grouped weight-gradient GEMM), then their biases
      o.wqkv = add_dense(p + "self_attention/dense/kernel", {E, E}, L2);
      add_dense(p + "self_attention/dense_1/kernel", {E, E}, L2);
      add_dense(p + "self_attention/dense_2/kernel", {E, E}, L2);
      o.bqkv = add_dense(p + "self_attention/dense/bias", {E}, L2);
      add_dense(p + "self_attention/dense_1/bias", {E}, L2);
      add_dense(p + "self_attention/dense_2/bias", {E}, L2);
      o.ln_a_beta = add_dense(p + "ln/Variable", {E}, L2);
      o.ln_a_gamma = add_dense(p + "ln/Variable_1", {E}, L2);
      o.w1 = add_dense(p + "multihead_attention/conv1d/kernel", {1, E, E}, L2);
      o.w2 = add_dense(p + "multihead_attention/conv1d_1/kernel", {1, E, E}, L2);
      o.b1 = add_dense(p + "multihead_attention/conv1d/bias", {E}, L2);
      o.b2 = add_dense(p + "multihead_attention/conv1d_1/bias", {E}, L2);
      o.ln_b_beta = add_dense(p + "ln_1/Variable", {E}, L2);
      o.ln_b_gamma = add_dense(p + "ln_1/Variable_1", {E}, L2);
    }
    for (int i = 0; i < BN_COUNT; ++i) bnoff[i] = BnOff{0, 0, 0, 0, 0};
    tower_in = 2 * E;
    tower = add_mlp({"sequential/logit_fcn"}, {L2}, tower_in, 100, 64, true, &bnoff[BN_T0], &bnoff[BN_T1]);   // sequential_base_model.py:76-79
    // ---- workspace
    add_ws("sib.ids_item", PAMREC_I32, {2, N});      // satisfied-only ids (looked up), then the full-history ids (L2 rows only)
    add_ws("sib.ids_cate", PAMREC_I32, {2, N});
    add_ws("sib.h", PAMREC_F32, {2, N, E});
    add_ws("tgt", PAMREC_F32, {B, E});
    add_ws("x0", PAMREC_F32, {N, E});               // history token + position row
    for (int b = 0; b < 2; ++b) {
      const std::string p = "blk" + std::to_string(b) + ".";
      add_ws(p + "xq", PAMREC_F32, {N, 2 * E});     // LN(x) | x
      add_ws(p + "qkv", PAMREC_F32, {N, 3 * E});
      add_ws(p + "ml", PAMREC_F32, {N, 2});
      add_ws(p + "y", PAMREC_F32, {N, E});
      add_ws(p + "f", PAMREC_F32, {N, E});          // LN_1(y)
      add_ws(p + "hpre", PAMREC_F32, {N, E});       // f W1 + b1 (the ReLU pattern of the point-wise FFN)
      add_ws(p + "out", PAMREC_F32, {N, E});
    }
    add_ws("u", PAMREC_F32, {B, 2 * E});            // final state | target
    add_ws("zt0", PAMREC_F32, {B, 100});
    add_ws("zt1", PAMREC_F32, {B, 64});
    add_ws("logits", PAMREC_F32, {B, 1});
    add_ws("losses", PAMREC_F32, {8});
    add_ws("loss_acc", PAMREC_F64, {8});
    add_ws("d_logits", PAMREC_F32, {B, 1});
    add_ws("d_t1", PAMREC_F32, {B, 64});
    add_ws("d_t0", PAMREC_F32, {B, 100});
    add_ws("d_u", PAMREC_F32, {B, 2 * E});
    add_ws("d_tgt_total", PAMREC_F32, {B, E});
    add_ws("sas.g_a", PAMREC_F32, {N, E});          // gradient of a block's output (ping)
    add_ws("sas.g_b", PAMREC_F32, {N, E});          // ... (pong)
    add_ws("sas.hid", PAMREC_F32, {N, E});
    add_ws("sas.d_hpre", PAMREC_F32, {N, E});
    add_ws("sas.d_y", PAMREC_F32, {N, E});
    add_ws("sas.d_qkv", PAMREC_F32, {N, 3 * E});
    add_ws("sas.dq", PAMREC_F32, {N});
    add_ws("sib.dh", PAMREC_F32, {2, N, E});        // [0] = gradient of x0 = rows of the satisfied lookups; [1] = 0 (L2 rows only)
    add_ws("sib.has0", PAMREC_I32, {4});
    add_bn_ws();
    add_optim_ws();
    const int64_t NK = 2 * N + B;
    cub_keys_table = NK;
    for (const char* t : {"item", "cate"}) {
      std::string p = std::string("sp.") + t + ".";
      for (const char* n : {"keys", "idx", "skeys", "sidx", "uidx", "ukeys"}) add_ws(p + n, PAMREC_I32, {NK});
      add_ws(p + "slot", PAMREC_I32, {t[0] == 'i' ? n_items : n_cates});
      add_ws(p + "accum", PAMREC_F32, {NK, t[0] == 'i' ? item_dim : cate_dim});
    }
    add_ws("sp.nuniq", PAMREC_I32, {8});
    add_ws("dp.scalars", PAMREC_F64, {8});
    cub_keys = NK;
    add_ws("cub_temp", PAMREC_U8, {(int64_t)(16u << 20) + 16 * cub_keys});
    (void)c;
  }

  void build(const PamrecConfig& c) {
    n_users = c.n_users; n_items = c.n_items; n_cates = c.n_cates; T = c.max_seq_len; Bcap = c.max_batch;
    world = c.world_size < 1 ? 1 : c.world_size; table_mode = c.table_mode;
    model_kind = c.model_kind;
    item_dim = c.item_dim ? c.item_dim : kI; cate_dim = c.cate_dim ? c.cate_dim : kC; user_dim = c.user_dim ? c.user_dim : PAMREC_USER_DIM;
    emb_dim = item_dim + cate_dim;
    if (model_kind == PAMREC_MODEL_SASREC) { build_sasrec(c); return; }
    if (model_kind != PAMREC_MODEL_PAMREC) { build_sibling(c); return; }
    const int L2 = PAMREC_SEG_L2;
    // ---- dense pool: encoder first so that every float4-loaded matrix starts on a 16-byte boundary
    pos = add_dense("sequential/embedding/position_embedding", {T, kD}, PAMREC_SEG_POS);
    for (int b = 0; b < 2; ++b) {
      std::string p = "sequential/pamrec/num_blocks_" + std::to_string(b) + "/";
      BlockOff& o = blk[b];
      o.ln_a_beta = add_dense(p + "ln/Variable", {kD}, L2);
      o.ln_a_gamma = add_dense(p + "ln/Variable_1", {kD}, L2);
      o.wq = add_dense(p + "self_attention/Q_timeaware_embedding", {kNB, kDD}, L2);
      o.wk = add_dense(p + "self_attention/K_timeaware_embedding", {kNB, kDD}, L2);
      o.wv = add_dense(p + "self_attention/V_timeaware_embedding", {kNB, kDD}, L2);
      o.w1 = add_dense(p + "multihead_attention/conv1d/kernel", {1, kD, kD}, L2);
      o.b1 = add_dense(p + "multihead_attention/conv1d/bias", {kD}, L2);
      o.w2 = add_dense(p + "multihead_attention/conv1d_1/kernel", {1, kD, kD}, L2);
      o.b2 = add_dense(p + "multihead_attention/conv1d_1/bias", {kD}, L2);
      o.ln_b_beta = add_dense(p + "ln_1/Variable", {kD}, L2);
      o.ln_b_gamma = add_dense(p + "ln_1/Variable_1", {kD}, L2);
    }
    score = add_mlp({"sequential/pamrec/new_long/score_1"}, {L2}, kD, 20, 1, false, &bnoff[BN_S0], &bnoff[BN_S1]);
    std::vector<std::string> ex;
    for (int j = 0; j < 5; ++j) ex.push_back("sequential/pamrec/expert_" + std::to_string(j));
    expert = add_mlp(ex, {L2, L2, L2, L2, L2}, kD, 100, 64, false, &bnoff[BN_E0], &bnoff[BN_E1]);
    gate = add_mlp({"sequential/pamrec/gate_main", "sequential/pamrec/gate_sub"}, {L2, L2}, kD, 64, 5, false,
                   &bnoff[BN_G0], &bnoff[BN_G1]);
    tower = add_mlp({"sequential/logit_fcn", "sequential/valid_logit_fcn", "xilidu_logit_fcn"}, {L2, L2, 0}, 64 + kE, 100, 64,
                    true, &bnoff[BN_T0], &bnoff[BN_T1]);
    // dead-for-logits branches (pamrec.py:293-311): variables exist, receive only the L2 gradient
    const char* dead[3] = {"new_distill", "long_term", "short_term"};
    const int dq[3] = {40, 20, 20};
    for (int i = 0; i < 3; ++i) {
      std::string p = std::string("sequential/pamrec/") + dead[i] + "/attention_fcn";
      add_dense(p + "/attention_mat", {kD, dq[i]}, L2 | PAMREC_SEG_DEAD);
      add_mlp({p + "/att_fcn"}, {L2 | PAMREC_SEG_DEAD}, 4 * dq[i], 80, 40, true, nullptr, nullptr, false);
    }

    // ---- workspace
    const int64_t B = Bcap, N = (int64_t)Bcap * T;
    const int64_t NT = N / kTokTile + kNB + 2;   // bucket-sorted tiles
    add_ws("bucket", PAMREC_I32, {N});
    add_ws("perm", PAMREC_I32, {N});
    add_ws("bucket_ctl", PAMREC_I32, {64});       // [0..15] counts, [16..31] cursors, [32] n_tiles
    add_ws("tile_bucket", PAMREC_I32, {NT});
    add_ws("tile_begin", PAMREC_I32, {NT});
    add_ws("tile_count", PAMREC_I32, {NT});
    add_ws("x0", PAMREC_F32, {B, T, kD});
    add_ws("tgt", PAMREC_F32, {B, kE});
    for (int b = 0; b < 2; ++b) {
      std::string p = "blk" + std::to_string(b) + ".";
      // pv: the attention output before the residual, P V = y - qin, kept apart because |qin| ~ 100 |P V|: the backward's
      // D = dY . (P V) taken from y - qin lost 8 bits (1e-4 of dQ, dK), which TF's softmax gradient does not
      for (const char* n : {"qin", "Q", "K", "V", "y", "pv", "out"}) add_ws(p + n, PAMREC_F32, {B, T, kD});
      add_ws(p + "ml", PAMREC_F32, {B, T, 2});   // softmax row maximum and row sum, kept for the backward pass
    }
    add_ws("z1", PAMREC_F32, {B, T, 20});
    add_ws("z2", PAMREC_F32, {B, T});
    add_ws("pool.aw", PAMREC_F32, {B, T});        // attention-pooling weights, kept for the backward pass (kernels_head2.cu)
    add_ws("head.wT", PAMREC_F32, {3 * 6400 + 3 * 8400 + 5 * 6400 + 2 * 320 + 628 * 40});   // transposed head weights of the dX chain
    add_ws("new_long", PAMREC_F32, {B, kD});
    add_ws("ze0", PAMREC_F32, {B, 500});
    add_ws("zg0", PAMREC_F32, {B, 128});
    add_ws("ze1", PAMREC_F32, {B, 320});
    add_ws("zg1", PAMREC_F32, {B, 10});
    add_ws("u", PAMREC_F32, {B, 168});
    add_ws("zt0", PAMREC_F32, {B, 300});
    add_ws("zt1", PAMREC_F32, {B, 192});
    add_ws("logits", PAMREC_F32, {B, 3});
    add_ws("losses", PAMREC_F32, {8});
    add_ws("loss_acc", PAMREC_F64, {8});          // [0] data [1] aux [2] order [3] regular
    // gradients
    add_ws("d_logits", PAMREC_F32, {B, 3});
    add_ws("d_t1", PAMREC_F32, {B, 192});
    add_ws("d_t0", PAMREC_F32, {B, 300});
    add_ws("d_u", PAMREC_F32, {B, 168});
    add_ws("d_e1", PAMREC_F32, {B, 320});
    add_ws("d_g1", PAMREC_F32, {B, 10});
    add_ws("d_e0", PAMREC_F32, {B, 500});
    add_ws("d_g0", PAMREC_F32, {B, 128});
    add_ws("d_new_long", PAMREC_F32, {B, kD});
    add_ws("d_tgt", PAMREC_F32, {B, kE});
    add_ws("d_tgt_total", PAMREC_F32, {B, kE});
    add_ws("d_z2", PAMREC_F32, {B, T});
    add_ws("d_a1", PAMREC_F32, {B, T, 20});
    add_ws("g_a", PAMREC_F32, {B, T, kD});        // ping-pong grads of block outputs / inputs
    add_ws("g_b", PAMREC_F32, {B, T, kD});
    add_ws("d_y", PAMREC_F32, {B, T, kD});
    add_ws("d_Q", PAMREC_F32, {B, T, kD});
    add_ws("d_K", PAMREC_F32, {B, T, kD});
    add_ws("d_V", PAMREC_F32, {B, T, kD});
    // inputs of the blocks' weight gradients (launch_enc_dw, side stream), which may still be reading them while the main stream
    // runs the next block's backward: block 1 keeps its own dQ, dK, dV and a copy of its output gradient (d_Q, d_K, d_V and
    // g_a are block 0's by then); h = relu(f W1 + b1) and dH o relu' of both blocks
    for (const char* n : {"blk1.d_Q", "blk1.d_K", "blk1.d_V", "blk1.d_out"}) add_ws(n, PAMREC_F32, {B, T, kD});
    for (const char* n : {"blk0.h", "blk0.dhr", "blk1.h", "blk1.dhr"}) add_ws(n, PAMREC_F32, {B, T, kD});
    // batch-norm statistics, optimiser scratch
    add_bn_ws();
    add_optim_ws();
    // sparse path: keys = history ids then target ids.  "sp.*" is the plan of THIS rank's lookups; the slot map
    // (table row -> unique index) always covers the rows this rank owns.
    const int64_t NK = N + B;
    const bool sharded = table_mode == PAMREC_TABLES_SHARDED;
    cub_keys_table = NK;
    for (const char* t : {"item", "cate"}) {
      std::string p = std::string("sp.") + t + ".";
      if (sharded) {
        add_ws(p + "keys", PAMREC_I32, {NK});
        add_ws(p + "idx", PAMREC_I32, {NK});
        add_ws(p + "skeys", PAMREC_I32, {NK});
        add_ws(p + "sidx", PAMREC_I32, {NK});
        add_ws(p + "uidx", PAMREC_I32, {NK});
        add_ws(p + "slot", PAMREC_I32, {rows_of(t[0] == 'i' ? n_items : n_cates)});
      }
      add_ws(p + "ukeys", PAMREC_I32, {NK});
      add_ws(p + "accum", PAMREC_F32, {NK, t[0] == 'i' ? kI : kC});
    }
    if (sharded) {
      add_ws("sp.user.keys", PAMREC_I32, {B});
      add_ws("sp.user.idx", PAMREC_I32, {B});
      add_ws("sp.user.skeys", PAMREC_I32, {B});
      add_ws("sp.user.sidx", PAMREC_I32, {B});
      add_ws("sp.user.uidx", PAMREC_I32, {B});
      add_ws("sp.user.slot", PAMREC_I32, {rows_of(n_users)});
    }
    add_ws("sp.user.ukeys", PAMREC_I32, {B});
    add_ws("sp.nuniq", PAMREC_I32, {8});           // 0 item 1 cate 2 user ; 4 5 6 = owner-side plans (sharded tables)
    add_ws("dp.scalars", PAMREC_F64, {8});         // [0] listwise groups with a non-zero label sum over all ranks
    cub_keys = NK;
    if (!sharded) {
      // whole tables on this GPU (kernels_sparse2.cu): ONE plan over the lookups of the three id spaces
      const int64_t NKA = 2 * NK + B;
      for (const char* n : {"keys", "idx", "skeys", "sidx", "uidx"}) add_ws(std::string("sp2.") + n, PAMREC_I32, {NKA});
      add_ws("sp2.meta", PAMREC_I32, {16});
      add_ws("sp2.slot", PAMREC_I32, {(int64_t)n_items + n_cates + n_users});
      add_ws("sp2.dflag", PAMREC_I32, {2 * NK});
      add_ws("sp2.l2sq", PAMREC_F64, {4});
      if (table_mode == PAMREC_TABLES_REPLICATED && world > 1)
        add_ws("rep.grad", PAMREC_F32, {(int64_t)n_items * 17 + (int64_t)n_cates * 5 + n_users});
      cub_keys = NKA;
    }
    if (table_mode == PAMREC_TABLES_SHARDED) {
      // exchange buffers ("sh.*") and the owner-side plan of the rows other ranks asked this rank for ("so.*")
      auto dim = [&](int64_t vocab, int64_t nk, int width) {
        ShardDim d;
        d.vocab = vocab; d.rps = rows_of(vocab); d.nk = nk; d.width = width;
        d.cap_recv = (int64_t)world * (nk < d.rps ? nk : d.rps);   // a rank can ask for at most min(nk, rps) distinct rows
        return d;
      };
      sh_item = dim(n_items, NK, kI); sh_cate = dim(n_cates, NK, kC); sh_user = dim(n_users, B, 0);
      const ShardDim* dims[3] = {&sh_item, &sh_cate, &sh_user};
      const char* names[3] = {"item", "cate", "user"};
      for (int i = 0; i < 3; ++i) {
        const ShardDim& d = *dims[i];
        std::string p = std::string("sh.") + names[i] + ".", q = std::string("so.") + names[i] + ".";
        add_ws(p + "inv", PAMREC_I32, {d.nk});
        add_ws(p + "send_ids", PAMREC_I32, {d.nk});
        add_ws(p + "off", PAMREC_I32, {128});
        add_ws(p + "recv_ids", PAMREC_I32, {d.cap_recv});
        if (d.width) {
          add_ws(p + "rows", PAMREC_F32, {d.nk, d.width});          // rows received from their owners (forward)
          add_ws(p + "xrows", PAMREC_F32, {d.cap_recv, d.width});   // owner: rows served (forward) / row gradients received
          add_ws(q + "accum", PAMREC_F32, {d.cap_recv, d.width});
        }
        for (const char* n : {"keys", "idx", "skeys", "sidx", "uidx", "ukeys"}) add_ws(q + n, PAMREC_I32, {d.cap_recv});
        if (d.cap_recv > cub_keys) cub_keys = d.cap_recv;
      }
      add_ws("sh.counts_send", PAMREC_I32, {(int64_t)world * 4});
      add_ws("sh.counts_recv", PAMREC_I32, {(int64_t)world * 4});
      add_ws("sh.scratch", PAMREC_F64, {8});
    }
    add_ws("cub_temp", PAMREC_U8, {(int64_t)(16u << 20) + 16 * cub_keys});
  }
};

}  // namespace pamrec
