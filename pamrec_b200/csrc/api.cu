// C ABI of libpamrec_b200.so (see include/pamrec_b200.h): handle, inventory queries and the
// orchestration of one train / score step as a sequence of kernel launches on the caller's stream.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <algorithm>
#include <cstdlib>
#include <functional>
#include <string>
#include <vector>

#include "comm.h"
#include "head2.h"
#include "kernels.h"
#include "layout.h"

using namespace pamrec;

// host view of one table's all-to-all for the current batch (element = one id / one row)
struct Xchg {
  std::vector<int64_t> soff, scnt, roff, rcnt;
  int64_t n_send = 0, n_recv = 0;
};

// One id space (layout.h: IdSpace) bound to the workspace and the caller's tables by pamrec_bind.
struct IdTables {
  const IdSpace* d = nullptr;
  SparseTable req;           // plan of this rank's lookups ("sp.<name>.*")
  SparseTable own;           // sharded: plan of the rows the other ranks asked this rank for ("so.<name>.*"), on the local shard
  SparseTable tab[2];        // the parameter tables, each on the plan of its update (own when sharded, else req)
  const int* sib_ids;        // siblings: the history lookups of a batch, written by the gather ("sib.ids_<name>")
  int* inv; int* send_ids; int* off; int* recv_ids; float* rows; float* xrows;   // sharded: the exchange ("sh.<name>.*")
  Xchg x;                    // sharded: the exchange of the current batch
};

struct PamrecHandle_ {
  PamrecConfig cfg;
  Layout L;
  PamrecBuffers buf;
  bool bound = false;
  int debug = 0;                // PAMREC_DEBUG_* test hooks
  std::string err;
  int64_t launches = 0;
  Prof prof;
  BnSet bn[BN_COUNT];
  std::vector<int> h_seg_id, h_seg_tab;
  Comm comm;
  int* h_counts = nullptr;      // pinned [2][world][4]: send | recv counts of the current batch (sharded tables)
  IdTables sp[3];               // L.idsp bound: item, cate, user
  bool xc_users = false;        // the current exchange carried user ids (training)
  bool sharded() const { return cfg.table_mode == PAMREC_TABLES_SHARDED; }
  bool sibling() const { return cfg.model_kind != PAMREC_MODEL_PAMREC; }
  bool replicated() const { return cfg.table_mode == PAMREC_TABLES_REPLICATED && cfg.world_size > 1; }
  // Internal side stream: work that is off the critical path of a step (the id sort of the sparse plan, the weight-gradient
  // GEMMs of the head) is forked from the caller's stream with events and joined back before anything consumes it.
  cudaStream_t side = nullptr;
  cudaEvent_t ev_side[16] = {};
  cudaEvent_t ev_join = nullptr, ev_plan = nullptr, ev_bucket = nullptr;
  int ev_next = 0;
  const void* plan_for = nullptr;   // batch whose sparse plan is in flight / ready on the side stream (local tables)
  int plan_rows = -1;
  // peer-memory mailboxes (kernels.h: p2p_mailbox_bytes): error word | persistent head exchanges | gradient exchange
  void* mbox = nullptr;
  void* mbox_peer[kP2PMaxWorld] = {};
  bool mbox_open = false;
  // persistent cooperative head kernels (kernels_head2.cu): barrier words, trace stamps
  unsigned* head_bar = nullptr;      // 64 words of barrier state, then 2 x 32 trace stamps (forward, backward)
  bool head_trace = false;
  unsigned long long* head_trace_cta = nullptr;   // debug: arrival stamps of every CTA at every barrier (2 kernels x 16 x 256)
  uint32_t coop_epoch = 0;          // mailbox epoch of the cooperative kernels (one per launch, all ranks in lockstep)
  // row-stationary persistent head kernels (kernels_head2.cu): the default; PAMREC_HEAD_LEGACY=1 (or a device without
  // cooperative launch, or more than 8 ranks) selects the stand-alone kernels of kernels_head.cu
  Head2 head2;
  int head2_grid = 0;
  bool use_head2() const { return head2_grid > 0 && (cfg.world_size == 1 || mbox_open); }
  uint32_t* mbox_err() const { return static_cast<uint32_t*>(mbox); }
  // gradient exchange through peer memory (kernels_p2p.cu:k_xr_*): dense gradients, then the replicated tables' gradient tables
  int64_t xr_dense() const { return (L.dense_numel + 63) / 64 * 64; }
  int64_t xr_floats() const { return xr_dense() + (replicated() ? sp2_rep_floats(cfg.n_items, cfg.n_cates, cfg.n_users) : 0); }
  char* xr_region(int p) const { return static_cast<char*>(mbox_peer[p]) + p2p_xr_offset(cfg.world_size); }
  bool use_xr() const { return mbox_open && cfg.world_size > 1; }
  uint32_t xr_epoch = 0;
  // the replicated tables' gradient tables + touch counts: inside the exchange buffers when those exist (the run walk writes
  // the contribution in place, the Adam sweep reads the reduced copy), else a workspace tensor reduced by NCCL
  float* rep_grad_in() const { return use_xr() ? xr_xbuf(xr_region(cfg.rank)) + xr_dense() : wf("rep.grad"); }
  float* rep_grad_out() const {
    return use_xr() ? xr_xbuf(xr_region(cfg.rank)) + p2p_xr_cap(cfg.world_size, xr_floats()) + xr_dense() : wf("rep.grad");
  }
  ~PamrecHandle_() {
    if (h_counts) cudaFreeHost(h_counts);
    for (int p = 0; p < kP2PMaxWorld; ++p)
      if (mbox_peer[p] && mbox_peer[p] != mbox) cudaIpcCloseMemHandle(mbox_peer[p]);
    if (mbox) cudaFree(mbox);
    if (head_bar) cudaFree(head_bar);
    if (head_trace_cta) cudaFree(head_trace_cta);
    for (auto e : ev_side) if (e) cudaEventDestroy(e);
    if (ev_join) cudaEventDestroy(ev_join);
    if (ev_plan) cudaEventDestroy(ev_plan);
    if (ev_bucket) cudaEventDestroy(ev_bucket);
    if (side) cudaStreamDestroy(side);
  }
  // run fn(side) after everything enqueued on `main` so far
  template <typename F>
  void fork(cudaStream_t main, F fn) {
    cudaEvent_t e = ev_side[ev_next];
    ev_next = (ev_next + 1) % 16;
    cudaEventRecord(e, main);
    cudaStreamWaitEvent(side, e, 0);
    fn(side);
  }
  void join(cudaStream_t main) {
    cudaEventRecord(ev_join, side);
    cudaStreamWaitEvent(main, ev_join, 0);
  }

  float* P(int64_t off) const { return buf.dense_param + off; }
  float* G(int64_t off) const { return buf.dense_grad + off; }
  template <typename T>
  T* ws(const std::string& name) const { return reinterpret_cast<T*>(static_cast<char*>(buf.workspace) + L.ws_off(name)); }
  float* wf(const std::string& name) const { return ws<float>(name); }
  int* wi(const std::string& name) const { return ws<int>(name); }
  double* wd(const std::string& name) const { return ws<double>(name); }
};

// binds the handle's launch accounting to this thread for the duration of one API call
struct ProfBind {
  PamrecHandle h; int64_t l0; Prof* prev;
  explicit ProfBind(PamrecHandle hh) : h(hh), l0(hh->prof.launches), prev(g_prof) { g_prof = &hh->prof; }
  ~ProfBind() { h->launches = h->prof.launches - l0; g_prof = prev; }
};

static int fail(PamrecHandle h, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  return -1;
}
static int check_cuda(PamrecHandle h, const char* where) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(h, "%s: %s", where, cudaGetErrorString(e));
  return 0;
}

extern "C" {

const char* pamrec_version(void) { return "pamrec_b200 0.1 (sm_100a)"; }

int pamrec_abi_sizes(int64_t out[6]) {
  if (!out) return -1;
  out[0] = sizeof(PamrecConfig); out[1] = sizeof(PamrecBatch); out[2] = sizeof(PamrecBuffers);
  out[3] = sizeof(PamrecTensorInfo); out[4] = sizeof(PamrecLines); out[5] = sizeof(PamrecVocab);
  return 0;
}

int pamrec_create(const PamrecConfig* cfg, PamrecHandle* out) {
  if (!cfg || !out) return -1;
  *out = nullptr;
  if (cfg->n_users < 1 || cfg->n_items < 1 || cfg->n_cates < 1) return -2;
  if (cfg->max_seq_len < 1 || cfg->max_seq_len > PAMREC_MAX_T) return -3;
  if (cfg->max_batch < 1) return -4;
  const int world = cfg->world_size < 1 ? 1 : cfg->world_size;
  if (world > 64 || cfg->rank < 0 || cfg->rank >= world) return -5;
  if (cfg->table_mode != PAMREC_TABLES_LOCAL && cfg->table_mode != PAMREC_TABLES_SHARDED && cfg->table_mode != PAMREC_TABLES_REPLICATED) return -6;
  if (world > 1 && cfg->table_mode == PAMREC_TABLES_LOCAL) return -6;        // multi-GPU = row-sharded or replicated tables
  if (cfg->table_mode != PAMREC_TABLES_SHARDED && (int64_t)cfg->n_items + cfg->n_cates + cfg->n_users >= ((int64_t)1 << 31)) return -7;
  if (cfg->loss_kind != PAMREC_LOSS_XENT && cfg->loss_kind != PAMREC_LOSS_SOFTMAX) return -8;
  if (cfg->loss_kind == PAMREC_LOSS_SOFTMAX) {
    const int g = cfg->softmax_group < 1 ? 1 : cfg->softmax_group;
    if (g > 1024 || (world > 1 && PAMREC_GROUP % g != 0)) return -8;
  }
  {
    // sharded keys are owner * rows_per_shard + local row: must fit an int32
    int64_t big = cfg->n_items > cfg->n_users ? cfg->n_items : cfg->n_users;
    if (cfg->n_cates > big) big = cfg->n_cates;
    if (((big + world - 1) / world) * world >= ((int64_t)1 << 31)) return -7;
  }
  if (cfg->model_kind < PAMREC_MODEL_PAMREC || cfg->model_kind > PAMREC_MODEL_SASREC) return -9;
  if (cfg->model_kind != PAMREC_MODEL_PAMREC && (world != 1 || cfg->table_mode != PAMREC_TABLES_LOCAL || cfg->loss_kind != PAMREC_LOSS_XENT))
    return -9;                                                               // sibling models: one GPU, whole tables, cross entropy
  const int di = cfg->item_dim ? cfg->item_dim : PAMREC_ITEM_DIM, dc = cfg->cate_dim ? cfg->cate_dim : PAMREC_CATE_DIM;
  const int du = cfg->user_dim ? cfg->user_dim : PAMREC_USER_DIM;
  if (!((di == 16 && dc == 4) || (di == 32 && dc == 8)) || !(du == 16 || du == 20 || du == 40)) return -10;
  if (cfg->model_kind == PAMREC_MODEL_PAMREC && (di != PAMREC_ITEM_DIM || dc != PAMREC_CATE_DIM || du != PAMREC_USER_DIM)) return -10;
  PamrecHandle h = new PamrecHandle_();
  h->cfg = *cfg;
  h->cfg.world_size = world;
  h->cfg.item_dim = di; h->cfg.cate_dim = dc; h->cfg.user_dim = du;
  if (h->cfg.softmax_group < 1) h->cfg.softmax_group = 1;
  h->L.build(h->cfg);
  const int n_seg = (int)h->L.dense.size();
  h->h_seg_id.assign((size_t)h->L.dense_numel, 0);
  h->h_seg_tab.assign((size_t)n_seg * 4, 0);
  for (int s = 0; s < n_seg; ++s) {
    const TensorDesc& t = h->L.dense[s];
    h->h_seg_tab[4 * s] = (int)t.offset;
    h->h_seg_tab[4 * s + 1] = (int)t.numel;
    h->h_seg_tab[4 * s + 2] = t.flags;
    for (int64_t i = 0; i < t.numel; ++i) h->h_seg_id[(size_t)(t.offset + i)] = s;
  }
  *out = h;
  return 0;
}

int pamrec_destroy(PamrecHandle h) {
  delete h;
  return 0;
}
const char* pamrec_last_error(PamrecHandle h) { return h ? h->err.c_str() : "null handle"; }
int64_t pamrec_dense_numel(PamrecHandle h) { return h ? h->L.dense_numel : -1; }
int64_t pamrec_bn_numel(PamrecHandle h) { return h ? h->L.bn_numel : -1; }
size_t pamrec_workspace_bytes(PamrecHandle h) { return h ? h->L.ws_bytes : 0; }
int64_t pamrec_last_launch_count(PamrecHandle h) { return h ? h->launches : -1; }
int64_t pamrec_shard_rows(PamrecHandle h, int64_t vocab_rows) { return h ? h->L.rows_of(vocab_rows) : -1; }

int pamrec_comm_unique_id(const char* nccl_path, char id_out[PAMREC_COMM_ID_BYTES]) {
  std::string err;
  if (Comm::unique_id(nccl_path, id_out, &err)) { fprintf(stderr, "pamrec_comm_unique_id: %s\n", err.c_str()); return -1; }
  return 0;
}
int pamrec_comm_init(PamrecHandle h, const char* nccl_path, const char id[PAMREC_COMM_ID_BYTES]) {
  if (!h || !id) return -1;
  if (h->comm.init(nccl_path, id, h->cfg.world_size, h->cfg.rank)) { h->err = "comm_init: " + h->comm.err; return -1; }
  return 0;
}
int pamrec_comm_mailbox_create(PamrecHandle h, char handle_out[PAMREC_IPC_HANDLE_BYTES]) {
  if (!h || !handle_out) return -1;
  static_assert(sizeof(cudaIpcMemHandle_t) == PAMREC_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t is 64 bytes");
  if (h->cfg.world_size > kP2PMaxWorld) return fail(h, "mailboxes support at most %d ranks", kP2PMaxWorld);
  if (!h->mbox) {
    const size_t bytes = p2p_mailbox_bytes(h->cfg.world_size, h->xr_floats());
    if (cudaMalloc(&h->mbox, bytes) != cudaSuccess) return check_cuda(h, "mailbox alloc");
    cudaMemset(h->mbox, 0, bytes);
    cudaDeviceSynchronize();
  }
  cudaIpcMemHandle_t ih;
  if (cudaIpcGetMemHandle(&ih, h->mbox) != cudaSuccess) return check_cuda(h, "cudaIpcGetMemHandle");
  memcpy(handle_out, &ih, sizeof ih);
  return 0;
}
int pamrec_comm_mailbox_open(PamrecHandle h, const char* handles) {
  if (!h || !handles || !h->mbox) return -1;
  for (int p = 0; p < h->cfg.world_size; ++p) {
    if (p == h->cfg.rank) { h->mbox_peer[p] = h->mbox; continue; }
    cudaIpcMemHandle_t ih;
    memcpy(&ih, handles + (size_t)p * PAMREC_IPC_HANDLE_BYTES, sizeof ih);
    void* ptr = nullptr;
    if (cudaIpcOpenMemHandle(&ptr, ih, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) return check_cuda(h, "cudaIpcOpenMemHandle");
    h->mbox_peer[p] = ptr;
  }
  h->mbox_open = true;
  return 0;
}
int pamrec_comm_destroy(PamrecHandle h) {
  if (!h) return -1;
  h->comm.destroy();
  return 0;
}

static const std::vector<TensorDesc>* pool_of(PamrecHandle h, int pool) {
  if (!h) return nullptr;
  if (pool == PAMREC_POOL_DENSE) return &h->L.dense;
  if (pool == PAMREC_POOL_BN) return &h->L.bn;
  if (pool == PAMREC_POOL_WORKSPACE) return &h->L.ws;
  return nullptr;
}
int pamrec_tensor_count(PamrecHandle h, int pool) {
  auto* v = pool_of(h, pool);
  return v ? (int)v->size() : -1;
}
int pamrec_tensor_info(PamrecHandle h, int pool, int index, PamrecTensorInfo* out) {
  auto* v = pool_of(h, pool);
  if (!v || !out || index < 0 || index >= (int)v->size()) return -1;
  const TensorDesc& t = (*v)[index];
  memset(out, 0, sizeof *out);
  snprintf(out->name, sizeof out->name, "%s", t.name.c_str());
  out->pool = t.pool; out->dtype = t.dtype; out->flags = t.flags;
  out->offset = t.offset; out->numel = t.numel; out->ndim = t.ndim;
  for (int i = 0; i < 4; ++i) out->shape[i] = t.shape[i];
  return 0;
}

// ------------------------------------------------------------------------------------------
static BnSet make_bn(PamrecHandle h, int id, const char* name) {
  const BnOff& o = h->L.bnoff[id];
  BnSet s;
  s.C = o.C;
  s.gamma = h->P(o.gamma); s.beta = h->P(o.beta);
  s.dgamma = h->G(o.gamma); s.dbeta = h->G(o.beta);
  s.mmean = h->buf.bn_moving + o.mm; s.mvar = h->buf.bn_moving + o.mv;
  std::string p = std::string("bn.") + name;
  s.sums = h->wd(p + ".sums"); s.stat = h->wf(p + ".stat"); s.bsums = h->wd("bn.bsums") + h->L.bn_bsums_off[id];
  return s;
}

static void bind_id_spaces(PamrecHandle h) {
  const PamrecBuffers& u = h->buf;
  float* const w[4] = {u.item_w, u.cate_w, u.ulong_w, u.ushort_w};
  float* const m[4] = {u.item_m, u.cate_m, u.ulong_m, u.ushort_m};
  float* const v[4] = {u.item_v, u.cate_v, u.ulong_v, u.ushort_v};
  int* nuniq = h->wi("sp.nuniq");
  double* normsq = h->wd("sp_normsq");
  for (int t = 0; t < h->L.n_idsp; ++t) {
    const IdSpace& d = h->L.idsp[t];
    IdTables& s = h->sp[t];
    s = IdTables{};
    s.d = &d;
    const std::string p = std::string("sp.") + d.name + ".", q = std::string("sh.") + d.name + ".", o = std::string("so.") + d.name + ".";
    SparseTable& r = s.req;
    r.width = d.width; r.n_rows = h->sharded() ? d.rows * h->cfg.world_size : d.rows;
    if (d.slot) {
      r.keys = h->wi(p + "keys"); r.idx = h->wi(p + "idx"); r.skeys = h->wi(p + "skeys"); r.sidx = h->wi(p + "sidx");
      r.uidx = h->wi(p + "uidx"); r.slot = h->wi(p + "slot");
    }
    r.ukeys = h->wi(p + "ukeys");
    if (d.accum) r.accum = h->wf(p + "accum");
    r.nuniq = nuniq + t; r.normsq = normsq + d.tab0;
    if (h->sibling() && d.accum) s.sib_ids = h->wi(std::string("sib.ids_") + d.name);
    if (h->sharded()) {
      SparseTable& a = s.own;
      a.width = d.width; a.n_rows = d.rows; a.slot = r.slot;
      a.keys = h->wi(o + "keys"); a.idx = h->wi(o + "idx"); a.skeys = h->wi(o + "skeys"); a.sidx = h->wi(o + "sidx");
      a.uidx = h->wi(o + "uidx"); a.ukeys = h->wi(o + "ukeys");
      if (d.accum) a.accum = h->wf(o + "accum");
      a.nuniq = nuniq + 4 + t;
      a.normsq = h->wd("sh.scratch");     // the un-deduplicated rows' norm is the requesters' (req.normsq)
      s.inv = h->wi(q + "inv"); s.send_ids = h->wi(q + "send_ids"); s.off = h->wi(q + "off"); s.recv_ids = h->wi(q + "recv_ids");
      if (d.accum) { s.rows = h->wf(q + "rows"); s.xrows = h->wf(q + "xrows"); }
    }
    for (int k = 0; k < d.n_tab; ++k) {
      SparseTable& e = s.tab[k];
      e = h->sharded() ? s.own : s.req;
      e.w = w[d.tab0 + k]; e.m = m[d.tab0 + k]; e.v = v[d.tab0 + k];
      e.normsq = normsq + d.tab0 + k;
      if (d.has0) e.l2_has0 = h->wi("sib.has0") + t;
    }
  }
}

static int build_head(PamrecHandle h, cudaStream_t st);
static HeadDyn head_dyn(PamrecHandle h, const PamrecBatch* b, bool training, int slot0);

int pamrec_bind(PamrecHandle h, const PamrecBuffers* bufs, void* stream) {
  if (!h || !bufs) return -1;
  cudaStream_t st = (cudaStream_t)stream;
  if (bufs->workspace_bytes < h->L.ws_bytes) return fail(h, "workspace too small: %zu < %zu", bufs->workspace_bytes, h->L.ws_bytes);
  if (!bufs->dense_param || !bufs->dense_grad || !bufs->dense_m || !bufs->dense_v || !bufs->bn_moving || !bufs->item_w ||
      !bufs->cate_w || !bufs->ulong_w || !bufs->ushort_w || !bufs->workspace)
    return fail(h, "null buffer");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(h, "no CUDA device: the CUDA path is the only path"); }
  h->buf = *bufs;
  if (init_encoder_kernels(h->cfg.max_seq_len)) return check_cuda(h, "shared-memory opt-in of the encoder kernels");
  if (h->cfg.model_kind == PAMREC_MODEL_SASREC && init_sas_kernels(h->cfg.max_seq_len))
    return check_cuda(h, "shared-memory opt-in of the SASRec attention kernels");
  if (init_attn_mma_kernels(h->cfg.max_seq_len)) return check_cuda(h, "shared-memory opt-in of the MMA attention kernels");
  if (!h->side) {
    if (cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) != cudaSuccess) return fail(h, "cannot create the side stream");
    for (auto& e : h->ev_side) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_plan, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_bucket, cudaEventDisableTiming);
  }
  static const char* names[BN_COUNT] = {"s0", "s1", "e0", "g0", "e1", "g1", "t0", "t1"};
  for (int i = 0; i < BN_COUNT; ++i) h->bn[i] = make_bn(h, i, names[i]);
  size_t need = sparse_temp_bytes(h->L.cub_keys);
  if (!h->sharded()) { const size_t n2 = sp2_temp_bytes(h->L.cub_keys); need = n2 > need ? n2 : need; }
  size_t have = (size_t)h->L.ws[h->L.ws_index["cub_temp"]].numel;
  if (need > have) return fail(h, "cub temp storage: need %zu have %zu", need, have);
  cudaMemsetAsync(h->buf.workspace, 0, h->L.ws_bytes, st);
  bind_id_spaces(h);
  for (int t = 0; t < h->L.n_idsp; ++t)
    if (h->L.idsp[t].slot) cudaMemsetAsync(h->sp[t].req.slot, 0xFF, (size_t)h->L.idsp[t].rows * 4, st);
  if (!h->sharded() && !h->sibling())
    cudaMemsetAsync(h->wi("sp2.slot"), 0xFF, ((size_t)h->cfg.n_items + h->cfg.n_cates + h->cfg.n_users) * 4, st);
  if (h->sharded() && !h->h_counts &&
      cudaMallocHost(&h->h_counts, sizeof(int) * (8 * (size_t)h->cfg.world_size + 4)) != cudaSuccess)
    return fail(h, "cudaMallocHost for the exchange counts failed");
  cudaMemcpyAsync(h->wi("seg_id"), h->h_seg_id.data(), h->h_seg_id.size() * 4, cudaMemcpyHostToDevice, st);
  cudaMemcpyAsync(h->wi("seg_tab"), h->h_seg_tab.data(), h->h_seg_tab.size() * 4, cudaMemcpyHostToDevice, st);
  if (h->sibling()) h->head2_grid = 0;                     // sibling models run on the stand-alone kernels (api_sibling.inl)
  else if (int rc = build_head(h, st)) return rc;
  cudaStreamSynchronize(st);
  h->bound = true;
  return check_cuda(h, "bind");
}

static int check_batch(PamrecHandle h, const PamrecBatch* b, bool training) {
  if (!h) return -1;
  if (!h->bound) return fail(h, "pamrec_bind has not been called");
  if (!b) return fail(h, "null batch");
  if (b->batch == 0 && (h->sharded() || h->cfg.world_size > 1)) return 0;  // this rank only takes part in the collectives
  if (b->batch < 1 || b->batch > h->cfg.max_batch) return fail(h, "batch %d outside [1, %d]", b->batch, h->cfg.max_batch);
  if (h->sibling()) {
    if (!b->satisfied_item_history || !b->satisfied_cate_history || !b->satisfied_mask || !b->item_history || !b->item_cate_history ||
        !b->mask || !b->items || !b->cates)
      return fail(h, "null batch field (the sibling models also read satisfied_item_history / satisfied_cate_history / satisfied_mask)");
    const bool sas = h->cfg.model_kind == PAMREC_MODEL_SASREC;
    if (training && (!b->labels_satisfied || (!sas && (!b->users || !b->labels_play)))) return fail(h, "null label field");
    return 0;
  }
  if (training && b->batch % PAMREC_GROUP != 0)
    return fail(h, "training batch %d is not a multiple of %d (pamrec.py:73-75)", b->batch, PAMREC_GROUP);
  if (training && h->cfg.loss_kind == PAMREC_LOSS_SOFTMAX && b->batch % h->cfg.softmax_group != 0)
    return fail(h, "training batch %d is not a multiple of the softmax group %d (base_model.py:224-225)", b->batch, h->cfg.softmax_group);
  if (!b->item_history || !b->item_cate_history || !b->item_loop_times_history || !b->mask || !b->items || !b->cates)
    return fail(h, "null batch field");
  if (training && (!b->users || !b->labels_satisfied || !b->labels_play || !b->plays)) return fail(h, "null label field");
  return 0;
}

// whole tables on this GPU (local or replicated): the one-sort plan / run walk of kernels_sparse2.cu
static Sp2 make_sp2(PamrecHandle h, const PamrecBatch* b) {
  Sp2 s;
  memset(&s, 0, sizeof s);
  const PamrecConfig& c = h->cfg;
  s.item_hist = b->item_history; s.cate_hist = b->item_cate_history; s.items = b->items; s.cates = b->cates; s.users = b->users;
  s.B = b->batch; s.N = (int64_t)b->batch * c.max_seq_len;
  s.n_items = c.n_items; s.n_cates = c.n_cates; s.n_users = c.n_users;
  s.keys = h->wi("sp2.keys"); s.idx = h->wi("sp2.idx"); s.skeys = h->wi("sp2.skeys"); s.sidx = h->wi("sp2.sidx"); s.uidx = h->wi("sp2.uidx");
  s.nuniq = h->wi("sp.nuniq"); s.meta = h->wi("sp2.meta");
  for (int t = 0; t < h->L.n_idsp; ++t) {
    const IdTables& x = h->sp[t];
    s.ukeys[t] = x.req.ukeys;
    if (x.d->accum) s.accum[t] = x.req.accum;
    for (int k = 0; k < x.d->n_tab; ++k) { s.w[x.d->tab0 + k] = x.tab[k].w; s.m[x.d->tab0 + k] = x.tab[k].m; s.v[x.d->tab0 + k] = x.tab[k].v; }
  }
  s.dflag[0] = h->wi("sp2.dflag"); s.dflag[1] = s.dflag[0] + h->L.idsp[0].nk;
  s.l2sq = h->wd("sp2.l2sq"); s.undedup = h->wd("sp_normsq");
  s.dX0 = h->wf("g_a"); s.dT = h->wf("d_tgt_total");
  if (h->replicated()) { s.mode = SP2_DENSE; s.rep_grad = h->rep_grad_in(); }
  else if (c.sparse_adam_mode == PAMREC_ADAM_LAZY) s.mode = SP2_FUSED;
  else { s.mode = SP2_COMPACT; s.slot = h->wi("sp2.slot"); }
  return s;
}
static AdamP make_adam(PamrecHandle h, float lr_t) {
  const PamrecConfig& c = h->cfg;
  AdamP a;
  a.lr = lr_t; a.b1 = c.beta1; a.b2 = c.beta2; a.eps = c.epsilon; a.l2 = c.embed_l2; a.clip = c.max_grad_norm; a.is_clip = c.is_clip_norm;
  a.lr_dev = nullptr;
  return a;
}

// Sparse update of one id space over the n lookups of plan p, in two halves: the sharded path all-reduces the clip norms between them.
// Reduce half: duplicate gradient rows summed into p.accum (when g: lookup i < n_hist reads row i of g->hist, the others row
// i - n_hist of g->tgt, from column g->col on), then the L2 rows of every parameter table.
struct GradRows { const float* hist; int hist_ld; const float* tgt; int tgt_ld; int col; };
static int sparse_reduce(PamrecHandle h, const SparseTable& p, int64_t n, int64_t n_hist, const GradRows* g, const SparseTable* tab,
                         int n_tab, cudaStream_t st) {
  if (g && launch_sparse_segreduce(p, n, n_hist, g->hist, g->hist_ld, g->col, g->tgt, g->tgt_ld, g->col, p.normsq, st))
    return fail(h, "no sparse kernels for table width %d", p.width);
  for (int k = 0; k < n_tab; ++k)
    if (launch_sparse_l2norm(tab[k], n, h->cfg.embed_l2, h->wd("loss_acc") + 3, st))
      return fail(h, "no sparse kernels for table width %d", tab[k].width);
  return 0;
}
// Apply half: Adam on every parameter table, then the slot map of their plan back to -1.
static int sparse_apply(PamrecHandle h, const SparseTable* tab, int n_tab, int64_t n, float lr_t, cudaStream_t st) {
  const PamrecConfig& c = h->cfg;
  for (int k = 0; k < n_tab; ++k)
    if (launch_sparse_adam(tab[k], n, c.sparse_adam_mode, c.embed_l2, lr_t, c.beta1, c.beta2, c.epsilon, c.max_grad_norm, c.is_clip_norm, st))
      return fail(h, "no sparse kernels for table width %d", tab[k].width);
  launch_slot_reset(tab[0], n, st);
  return 0;
}

// ------------------------------------------------------------------------------------------
// Row-sharded tables (PAMREC_TABLES_SHARDED): plan of this rank's lookups ("sp.*": keys are sharded-table addresses), exchange
// with the owners.

// ids of id space t (0 item, 1 cate, 2 user) that batch b looks up: history (users: the user ids), then targets (users: none)
static const int* hist_ids(const PamrecBatch* b, int t) { return t == 0 ? b->item_history : (t == 1 ? b->item_cate_history : b->users); }
static const int* tgt_ids(const PamrecBatch* b, int t) { return t == 0 ? b->items : (t == 1 ? b->cates : nullptr); }

// Forward half of the exchange: unique ids of the batch -> owners; owners' rows -> "sh.<table>.rows", one row per
// unique id, in the order of the plan's unique list ("sh.<table>.inv" maps every lookup position to its row).
// ONE host synchronisation: the per-peer counts must reach the host before the variable all-to-alls can be posted.
static int shard_exchange_fwd(PamrecHandle h, const PamrecBatch* b, bool training, cudaStream_t st) {
  const int W = h->cfg.world_size, B = b->batch, T = h->cfg.max_seq_len;
  void* tmp = h->ws<char>("cub_temp");
  const size_t tmp_bytes = (size_t)h->L.ws[h->L.ws_index.at("cub_temp")].numel;
  int* cs = h->wi("sh.counts_send");
  int* cr = h->wi("sh.counts_recv");
  cudaMemsetAsync(cs, 0, sizeof(int) * 4 * W, st);
  const int nt = training ? 3 : 2;                    // user ids travel when training only: their rows are L2 rows of the update
  h->xc_users = training;
  for (int t = 0; t < nt; ++t) {
    const IdTables& s = h->sp[t];
    const int64_t rps = s.d->rows, n = s.d->lookups(B, T), n_hist = s.d->n_hist(B, T);
    if (launch_sparse_plan(s.req, hist_ids(b, t), tgt_ids(b, t), n_hist, n - n_hist, W, rps, rps * W, false, tmp, tmp_bytes, st))
      return fail(h, "cub sort failed");
    launch_shard_route(s.req, n, W, rps, s.off, cs, t, s.send_ids, s.inv, st);
  }
  {
    PAMREC_PROF("xchg_counts", 1, st);
    if (h->comm.all_to_all(cs, cr, 4, COMM_I32, st)) return fail(h, "nccl: %s", h->comm.err.c_str());
    cudaMemcpyAsync(h->h_counts, cs, sizeof(int) * 4 * W, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(h->h_counts + 4 * W, cr, sizeof(int) * 4 * W, cudaMemcpyDeviceToHost, st);
    h->h_counts[8 * W] = 0;
    if (h->mbox_open) cudaMemcpyAsync(h->h_counts + 8 * W, h->mbox_err(), sizeof(int), cudaMemcpyDeviceToHost, st);
    if (cudaStreamSynchronize(st) != cudaSuccess) return check_cuda(h, "exchange counts");
    if (h->h_counts[8 * W]) return fail(h, "peer mailbox all-reduce timed out at sync point %d (a rank left the step?)", h->h_counts[8 * W] - 1);
  }
  for (int t = 0; t < 3; ++t) {
    Xchg& x = h->sp[t].x;
    x.soff.assign(W, 0); x.scnt.assign(W, 0); x.roff.assign(W, 0); x.rcnt.assign(W, 0);
    int64_t so = 0, ro = 0;
    for (int p = 0; p < W; ++p) {
      x.scnt[p] = t < nt ? h->h_counts[4 * p + t] : 0;
      x.rcnt[p] = t < nt ? h->h_counts[4 * W + 4 * p + t] : 0;
      x.soff[p] = so; so += x.scnt[p];
      x.roff[p] = ro; ro += x.rcnt[p];
    }
    x.n_send = so; x.n_recv = ro;
    if (ro > h->sp[t].d->cap_recv) return fail(h, "exchange overflow on table %s: %lld rows", h->sp[t].d->name, (long long)ro);
  }
  {
    PAMREC_PROF("xchg_ids", 1, st);
    int xrc = h->comm.group_start();                  // the group is closed on every path (comm.cu: close_group)
    for (int t = 0; t < nt && !xrc; ++t) {
      const IdTables& s = h->sp[t];
      xrc |= h->comm.all_to_all_v(s.send_ids, s.x.soff.data(), s.x.scnt.data(), s.recv_ids, s.x.roff.data(), s.x.rcnt.data(), 1, COMM_I32, st);
    }
    xrc |= h->comm.group_end();
    if (xrc) return fail(h, "nccl: %s", h->comm.err.c_str());
  }
  if (training) {
    // owner-side unique / slot plan of the rows other ranks asked for: needed by apply_gradients only, so it is sorted on the
    // side stream while the forward and backward passes run (the requester plans above are done with the cub scratch)
    int prc = 0;
    h->fork(st, [&](cudaStream_t s2) {
      for (const IdTables& s : h->sp)
        prc |= launch_sparse_plan(s.own, s.recv_ids, nullptr, s.x.n_recv, 0, 1, 0, s.own.n_rows, true, tmp, tmp_bytes, s2);
      cudaEventRecord(h->ev_plan, s2);
    });
    if (prc) return fail(h, "cub sort failed");
  }
  for (const IdTables& s : h->sp)
    if (s.d->accum) launch_serve_rows(s.tab[0].w, s.recv_ids, s.x.n_recv, s.d->width, s.xrows, st);
  {
    PAMREC_PROF("xchg_rows", 1, st);
    int xrc = h->comm.group_start();
    for (const IdTables& s : h->sp)
      if (s.d->accum && !xrc)
        xrc |= h->comm.all_to_all_v(s.xrows, s.x.roff.data(), s.x.rcnt.data(), s.rows, s.x.soff.data(), s.x.scnt.data(), s.d->width,
                                    COMM_F32, st);
    xrc |= h->comm.group_end();
    if (xrc) return fail(h, "nccl: %s", h->comm.err.c_str());
  }
  return 0;
}

// x0 / tgt of this rank's batch, from whole local tables or through the exchange
static int embed_forward(PamrecHandle h, const PamrecBatch* b, bool training, float* x0, cudaStream_t st) {
  const int B = b->batch, T = h->cfg.max_seq_len;
  if (!h->sharded()) {
    launch_embed_fwd(b->item_history, b->item_cate_history, b->items, b->cates, h->buf.item_w, h->buf.cate_w, h->P(h->L.pos), x0,
                     h->wf("tgt"), B, T, st);
    return 0;
  }
  if (int rc = shard_exchange_fwd(h, b, training, st)) return rc;
  const int64_t N = (int64_t)B * T;
  const IdTables& si = h->sp[0];
  const IdTables& sc = h->sp[1];
  launch_embed_fwd(si.inv, sc.inv, si.inv + N, sc.inv + N, si.rows, sc.rows, h->P(h->L.pos), x0, h->wf("tgt"), B, T, st);
  return 0;
}

int pamrec_gather_fwd(PamrecHandle h, const PamrecBatch* b, float* x0_out, void* stream) {
  if (int rc = check_batch(h, b, false)) return rc;
  if (h->sibling()) return fail(h, "pamrec_gather_fwd is PAMRec's fused gather; the sibling models gather inside pamrec_forward");
  ProfBind _pb(h);
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = embed_forward(h, b, false, x0_out ? x0_out : h->wf("x0"), st)) return rc;
  return check_cuda(h, "gather_fwd");
}

static DenseP dense_p(const float* X, int ldx, int M, int groups, int K, int N, const float* W, int ws, const float* bias,
                      int bs, float* Z, int ldz) {
  DenseP p;
  memset(&p, 0, sizeof p);
  p.X = X; p.ldx = ldx; p.M = M; p.n_groups = groups; p.K = K; p.N = N;
  p.W = W; p.w_stride = ws; p.bias = bias; p.b_stride = bs; p.Z = Z; p.ldz = ldz;
  return p;
}
static DenseDwP dw_p(const float* X, int ldx, int M, int groups, int K, int N, const float* dZ, int lddz, float* dW, int ws,
                     float* db, int bs) {
  DenseDwP p;
  memset(&p, 0, sizeof p);
  p.X = X; p.ldx = ldx; p.M = M; p.n_groups = groups; p.K = K; p.N = N; p.dZ = dZ; p.lddz = lddz;
  p.dW = dW; p.w_stride = ws; p.db = db; p.b_stride = bs;
  return p;
}
static DenseDxP dx_p(const float* dZ, int lddz, int M, int K, const float* Wbase, float* dX, int lddx, int accumulate) {
  DenseDxP p;
  memset(&p, 0, sizeof p);
  p.dZ = dZ; p.lddz = lddz; p.M = M; p.K = K; p.Wbase = Wbase; p.dX = dX; p.lddx = lddx; p.accumulate = accumulate;
  return p;
}
static void dx_add(DenseDxP& p, int slice, int out_off, int dz_off, int64_t w_off, int N) {
  if (slice >= p.n_slices) { p.n_slices = slice + 1; p.out_off[slice] = out_off; p.n_contrib[slice] = 0; }
  int c = p.n_contrib[slice]++;
  p.dz_off[slice][c] = dz_off; p.w_off[slice][c] = w_off; p.Ncon[slice][c] = N;
}

// One group-strided BN MLP (layout.h: MlpOff) bound to its buffers.  Layer 0 of member g reads the columns x_col[g].. of x
// (leading dimension ldx), layer l > 0 the member's own columns of z[l - 1]; layer l writes the member's columns g * n_of(l).. of
// z[l] (leading dimension width(l): pre-BN values, the output layer's logits).  dz[l], laid out like z[l], holds the gradient with
// respect to layer l's post-BN-ReLU activation (the output layer's: its logits).  The gradient of x goes to dx (leading dimension
// ldx), added to what dx holds when dx_acc: the gates add theirs to the experts'.
struct MlpBind {
  const MlpOff* m;
  int M; double count;                 // rows of this rank; rows that the batch norms normalise over (every rank's)
  const float* x; int ldx; int x_col[8];
  float* z[3]; float* dz[3];
  float* dx; int dx_acc;
};
using BnSync = std::function<void(const std::vector<int>&)>;
static void no_sync(const std::vector<int>&) {}

// Forward pass of MLPs that read the same input, layer by layer: one layer of every MLP, then (training) sync(ids) on the batch-norm
// sets that layer filled, then their statistics: e0, g0, finalize, e1, g1, finalize.
static void mlp_forward(PamrecHandle h, std::initializer_list<const MlpBind*> ms, bool training, const BnSync& sync, cudaStream_t st) {
  const MlpBind& first = **ms.begin();
  for (int l = 0; l < first.m->n_layers(); ++l) {
    std::vector<int> ids;
    for (const MlpBind* b : ms) {
      const MlpOff& m = *b->m;
      const int K = m.k_of(l), N = m.n_of(l);
      DenseP p = dense_p(l ? b->z[l - 1] : b->x, l ? m.width(l - 1) : b->ldx, b->M, m.G, K, N, h->P(m.w_of(l)), K * N,
                         h->P(m.b_of(l)), N, b->z[l], m.width(l));
      for (int g = 0; g < m.G; ++g) { p.x_off[g] = l ? g * K : b->x_col[g]; p.z_off[g] = g * N; }
      if (l) { const BnSet& in = h->bn[m.bn_of(l - 1)]; p.in_stat = in.stat; p.in_gamma = in.gamma; p.in_beta = in.beta; }
      if (l < 2 && training) { p.out_sums = h->bn[m.bn_of(l)].sums; ids.push_back(m.bn_of(l)); }
      launch_dense_fwd(p, st);
    }
    if (ids.empty()) continue;
    sync(ids);
    for (int id : ids) launch_bn_finalize(h->bn[id], first.count, st);
  }
}

// Backward pass of MLPs whose output gradients dz[top] are complete, layer by layer from the top.  Per MLP the weight gradient (no
// consumer before the optimiser: side stream) with the parameter gradients of its layer's batch norm (times g_scale), then the input
// gradient, which also accumulates the gradient sums of the batch norm below.  sync(ids) runs once those sums of the listed sets are
// complete: first for the top sets of MLPs without an output layer (their gradient comes from a pooling or mixing kernel; summed
// here by k_bn_bwd_stats), then after every layer but the first.
static void mlp_backward(PamrecHandle h, std::initializer_list<const MlpBind*> ms, float g_scale, const BnSync& sync, cudaStream_t st) {
  const BnSet* bn = h->bn;
  const MlpBind& first = **ms.begin();
  std::vector<int> ids;
  for (const MlpBind* b : ms)
    if (!b->m->out) { launch_bn_bwd_stats(bn[b->m->bn1], b->dz[1], b->z[1], b->M, st); ids.push_back(b->m->bn1); }
  if (!ids.empty()) sync(ids);
  for (int l = first.m->n_layers() - 1; l >= 0; --l) {
    ids.clear();
    for (const MlpBind* b : ms) {
      const MlpOff& m = *b->m;
      const int K = m.k_of(l), N = m.n_of(l);
      const int ldx = l ? m.width(l - 1) : b->ldx;
      DenseDwP w = dw_p(l ? b->z[l - 1] : b->x, ldx, b->M, m.G, K, N, b->dz[l], m.width(l), h->G(m.w_of(l)), K * N,
                        h->G(m.b_of(l)), N);
      DenseDxP x = dx_p(b->dz[l], m.width(l), b->M, K, h->buf.dense_param, l ? b->dz[l - 1] : b->dx, ldx, l ? 0 : b->dx_acc);
      for (int g = 0; g < m.G; ++g) {
        w.x_off[g] = l ? g * K : b->x_col[g]; w.z_off[g] = g * N;
        // one slice of dX per input column: the first member reading it opens the slice, later ones add to it in member order
        int s = 0;
        while (s < x.n_slices && x.out_off[s] != w.x_off[g]) ++s;
        dx_add(x, s, w.x_off[g], g * N, m.w_of(l) + (int64_t)g * K * N, N);
      }
      if (l) {
        const BnId id = m.bn_of(l - 1);
        w.in_stat = bn[id].stat; w.in_gamma = bn[id].gamma; w.in_beta = bn[id].beta;
        x.o = BnGradOut{b->z[l - 1], bn[id].stat, bn[id].gamma, bn[id].beta, bn[id].bsums};
        ids.push_back(id);
      }
      if (l < 2) {
        const BnId id = m.bn_of(l);
        w.g = x.g = BnGrad{b->z[l], bn[id].stat, bn[id].gamma, bn[id].beta, bn[id].bsums, b->count};
        w.g_dgamma = bn[id].dgamma; w.g_dbeta = bn[id].dbeta; w.g_C = bn[id].C; w.g_scale = g_scale;
      }
      h->fork(st, [&](cudaStream_t s2) { launch_dense_dw(w, s2); });
      launch_dense_dx(x, st);
    }
    if (!ids.empty()) sync(ids);
  }
}

// The stand-alone head's MLPs (pamrec.py:273 attention-pooling score, :26-50 experts and gates, :212-215 and :71 towers on main |
// target, sub | target, main | target) bound to their buffers.
struct HeadMlps { MlpBind score, expert, gate, tower; };
static HeadMlps head_mlps(PamrecHandle h, const PamrecBatch* b) {
  const Layout& L = h->L;
  const int B = b->batch, T = h->cfg.max_seq_len;
  const double Bg = b->global_batch > 0 ? b->global_batch : B * h->cfg.world_size;
  float* new_long = h->wf("new_long");
  float* d_new_long = h->wf("d_new_long");
  const int tin = L.tower.in;
  HeadMlps m;
  m.score = {&L.score, B * T, Bg * T, h->wf("blk1.out"), kD, {0}, {h->wf("z1"), h->wf("z2")}, {h->wf("d_a1"), h->wf("d_z2")},
             h->wf("g_a"), 1};
  m.expert = {&L.expert, B, Bg, new_long, kD, {0}, {h->wf("ze0"), h->wf("ze1")}, {h->wf("d_e0"), h->wf("d_e1")}, d_new_long, 0};
  m.gate = {&L.gate, B, Bg, new_long, kD, {0}, {h->wf("zg0"), h->wf("zg1")}, {h->wf("d_g0"), h->wf("d_g1")}, d_new_long, 1};
  m.tower = {&L.tower, B, Bg, h->wf("u"), 2 * tin, {0, tin, 0}, {h->wf("zt0"), h->wf("zt1"), h->wf("logits")},
             {h->wf("d_t0"), h->wf("d_t1"), h->wf("d_logits")}, h->wf("d_u"), 0};
  return m;
}

static int sib_forward(PamrecHandle h, const PamrecBatch* b, int training, float* pred_out, cudaStream_t st);
static int sib_backward(PamrecHandle h, const PamrecBatch* b, cudaStream_t st);
static int sib_apply(PamrecHandle h, const PamrecBatch* b, int64_t step, cudaStream_t st);
static int sas_forward(PamrecHandle h, const PamrecBatch* b, int training, float* pred_out, cudaStream_t st);
static int sas_backward(PamrecHandle h, const PamrecBatch* b, cudaStream_t st);
static int head_forward(PamrecHandle h, const PamrecBatch* b, bool training, float* pred_out, float* aw_out, cudaStream_t st);
static int pam_forward(PamrecHandle h, const PamrecBatch* b, int training, float* pred_out, bool keep_aw, cudaStream_t st);

int pamrec_forward(PamrecHandle h, const PamrecBatch* b, int training, float* pred_out, void* stream) {
  if (int rc = check_batch(h, b, training != 0)) return rc;
  ProfBind _pb(h);
  cudaStream_t st = (cudaStream_t)stream;
  if (h->cfg.model_kind == PAMREC_MODEL_SASREC) return sas_forward(h, b, training, pred_out, st);
  if (h->sibling()) return sib_forward(h, b, training, pred_out, st);
  return pam_forward(h, b, training, pred_out, false, st);
}

// PAMRec's forward pass; keep_aw (scoring, pamrec_attention): the head also leaves the pooling weights in "pool.aw"
static int pam_forward(PamrecHandle h, const PamrecBatch* b, int training, float* pred_out, bool keep_aw, cudaStream_t st) {
  const Layout& L = h->L;
  const int B = b->batch, T = h->cfg.max_seq_len, N = B * T;
  float* x0 = h->wf("x0");
  int* ctl = h->wi("bucket_ctl");
  // The bucket sort of the tokens depends on the play-ratio buckets of the batch only: on the side stream beside the gather
  // (whole tables; the sharded exchange synchronises with the host and keeps everything on one stream)
  const bool bucket_aside = !h->sharded();
  if (bucket_aside) {
    h->fork(st, [&](cudaStream_t s2) {
      launch_bucket_plan(b->item_loop_times_history, N, h->wi("bucket"), h->wi("perm"), ctl, h->wi("tile_bucket"), h->wi("tile_begin"),
                         h->wi("tile_count"), s2);
      cudaEventRecord(h->ev_bucket, s2);
    });
  }
  if (int rc = embed_forward(h, b, training != 0, x0, st)) return rc;
  if (training && !h->sharded() && B > 0) {
    // the id sort / unique pass of the sparse backward depends on the batch only: run it beside the forward pass
    int prc = 0;
    h->fork(st, [&](cudaStream_t s2) {
      prc |= launch_sp2_plan(make_sp2(h, b), h->ws<char>("cub_temp"), (size_t)L.ws[L.ws_index.at("cub_temp")].numel, s2);
      cudaEventRecord(h->ev_plan, s2);
    });
    if (prc) return fail(h, "cub sort failed");
    h->plan_for = b->item_history; h->plan_rows = B;
  }
  if (bucket_aside) cudaStreamWaitEvent(st, h->ev_bucket, 0);
  else launch_bucket_plan(b->item_loop_times_history, N, h->wi("bucket"), h->wi("perm"), ctl, h->wi("tile_bucket"),
                          h->wi("tile_begin"), h->wi("tile_count"), st);
  const int max_tiles = N / kTokTile + kNB + 1;   // at most one partial tile per bin: the 10 buckets and the zero bin
  const float* xin = x0;
  for (int k = 0; k < 2; ++k) {
    const BlockOff& o = L.blk[k];
    std::string p = "blk" + std::to_string(k) + ".";
    launch_proj_fwd(xin, h->wi("perm"), ctl, h->wi("tile_bucket"), h->wi("tile_begin"), h->wi("tile_count"), max_tiles,
                    h->P(o.wq), h->P(o.wk), h->P(o.wv), h->P(o.ln_a_beta), h->P(o.ln_a_gamma), h->wf(p + "qin"), h->wf(p + "Q"),
                    h->wf(p + "K"), h->wf(p + "V"), st);
    // the MMA kernel up to T = 128, the FFMA kernel beyond: attn_fwd per step on a B200 (1000 W) MMA vs FFMA 0.046 vs 0.066 ms on
    // takatak_b1025_t50, 0.078 vs 0.099 ms on wechat_b500_t100, 2.18 vs 1.45 ms on long_b4095_t200 (no T in between measured)
    if (T <= 128)
      launch_attn_fwd_mma(h->wf(p + "Q"), h->wf(p + "K"), h->wf(p + "V"), h->wf(p + "qin"), b->mask, h->wf(p + "y"), h->wf(p + "pv"), h->wf(p + "ml"), B, T, st);
    else
      launch_attn_fwd(h->wf(p + "Q"), h->wf(p + "K"), h->wf(p + "V"), h->wf(p + "qin"), b->mask, h->wf(p + "y"), h->wf(p + "pv"), h->wf(p + "ml"), B, T, st);
    float* hdbg = (training && (h->debug & PAMREC_DEBUG_SAVE_FFN_HIDDEN)) ? h->wf(k == 0 ? "d_Q" : "d_K") : nullptr;
    launch_ffn_fwd(h->wf(p + "y"), h->P(o.w1), h->P(o.b1), h->P(o.w2), h->P(o.b2), h->P(o.ln_b_beta), h->P(o.ln_b_gamma),
                   h->wf(p + "out"), hdbg, N, st);
    xin = h->wf(p + "out");
  }
  if (h->use_head2()) {
    // the whole head as ONE persistent cooperative kernel, row-stationary (kernels_head2.cu)
    HeadDyn d = head_dyn(h, b, training != 0, 0);
    d.pred = pred_out;
    d.keep_aw = keep_aw ? 1 : 0;
    if (launch_head2_fwd(h->head2, d, h->head2_grid, training ? "head_fwd" : "head_score", st)) return check_cuda(h, "cooperative head launch");
  } else if (int rc = head_forward(h, b, training != 0, pred_out, keep_aw ? h->wf("pool.aw") : nullptr, st)) {
    return rc;
  }
  return check_cuda(h, "forward");
}

// The stand-alone head (kernels_head.cu): a launch per layer.  Training: batch statistics of the listed sets -> (mean, invstd), moving
// averages; data parallel: the column sums (plus, once, the listwise-group count) are first summed over the ranks by NCCL.
// aw_out (nullable): the pooling weights are also written there.
static int head_forward(PamrecHandle h, const PamrecBatch* b, bool training, float* pred_out, float* aw_out, cudaStream_t st) {
  const int B = b->batch, T = h->cfg.max_seq_len;
  const int W = h->cfg.world_size;
  int crc = 0;
  bool with_scalars = true;            // the listwise-group count travels with the first sums
  auto sync_sums = [&](const std::vector<int>& ids) {
    if (W > 1 && !crc) {
      PAMREC_PROF("allreduce_bn_fwd", 1, st);
      crc |= h->comm.group_start();
      for (int id : ids) crc |= h->comm.all_reduce(h->bn[id].sums, 2 * (int64_t)h->bn[id].C, COMM_F64, st);
      if (with_scalars) crc |= h->comm.all_reduce(h->wd("dp.scalars"), 8, COMM_F64, st);
      crc |= h->comm.group_end();
    }
    with_scalars = false;
  };
  if (training && W > 1) {
    cudaMemsetAsync(h->wd("dp.scalars"), 0, 8 * sizeof(double), st);
    launch_count_valid_groups(b->plays, B, h->wd("dp.scalars"), st);
  }
  BnSet* bn = h->bn;
  if (!training) {
    for (int i = 0; i < BN_COUNT; ++i) launch_bn_eval_stat(bn[i], st);
  }
  const HeadMlps m = head_mlps(h, b);
  mlp_forward(h, {&m.score}, training, sync_sums, st);
  launch_pool_fwd(h->wf("blk1.out"), h->wf("z2"), bn[BN_S1], b->mask, h->wf("new_long"), aw_out, B, T, st);
  mlp_forward(h, {&m.expert, &m.gate}, training, sync_sums, st);
  launch_combine_fwd(h->wf("ze1"), h->wf("zg1"), bn[BN_E1], bn[BN_G1], h->wf("tgt"), h->wf("u"), B, st);
  mlp_forward(h, {&m.tower}, training, sync_sums, st);
  if (pred_out) launch_sigmoid_col0(h->wf("logits"), pred_out, B, st);
  if (crc) return fail(h, "nccl: %s", h->comm.err.c_str());
  return 0;
}

// ------------------------------------------------------------------------------------------
// per-call values of the cooperative head kernels; slot0 = first mailbox slot of this kernel's barriers
static HeadDyn head_dyn(PamrecHandle h, const PamrecBatch* b, bool training, int slot0) {
  HeadDyn d;
  memset(&d, 0, sizeof d);
  const int W = h->cfg.world_size;
  d.B = b->batch; d.T = h->cfg.max_seq_len; d.training = training ? 1 : 0; d.world = W; d.rank = h->cfg.rank;
  d.Bg = b->global_batch > 0 ? b->global_batch : b->batch * W;
  d.cntN = (double)d.Bg * d.T; d.cntB = (double)d.Bg;
  d.mask = b->mask; d.y_sat = b->labels_satisfied; d.y_play = b->labels_play; d.plays = b->plays;
  d.fuzhu_w = h->cfg.fuzhu_weight; d.order_w = h->cfg.order_weight;
  d.sm_group = h->cfg.loss_kind == PAMREC_LOSS_SOFTMAX ? h->cfg.softmax_group : 0;
  d.bar = h->head_bar;
  d.trace = h->head_trace ? reinterpret_cast<unsigned long long*>(h->head_bar + 64) + (slot0 ? 32 : 0) : nullptr;
  d.trace_cta = (h->head_trace && h->head_trace_cta) ? h->head_trace_cta + (slot0 ? 16 * 256 : 0) : nullptr;
  if (W > 1) {
    for (int p = 0; p < W; ++p) d.peer_ll[p] = reinterpret_cast<uint4*>(static_cast<char*>(h->mbox_peer[p]) + p2p_ll_offset());
    d.p2p_epoch = ++h->coop_epoch; d.p2p_slot0 = slot0; d.p2p_err = h->mbox_err();
  }
  return d;
}

// Pointers of the row-stationary head kernels (kernels_head2.cu); they never change after pamrec_bind.
static int build_head(PamrecHandle h, cudaStream_t st) {
  h->head2_grid = 0;
  if (getenv("PAMREC_HEAD_LEGACY") != nullptr) return 0;
  if (h->cfg.world_size > kP2PMaxWorld) return 0;
  const Layout& L = h->L;
  Head2& H = h->head2;
  memset(&H, 0, sizeof H);
  H.H = h->wf("blk1.out"); H.tgt = h->wf("tgt");
  H.s_w0 = h->P(L.score.w0); H.s_b0 = h->P(L.score.b0); H.s_w1 = h->P(L.score.w1); H.s_b1 = h->P(L.score.b1);
  H.e_w0 = h->P(L.expert.w0); H.e_b0 = h->P(L.expert.b0); H.e_w1 = h->P(L.expert.w1); H.e_b1 = h->P(L.expert.b1);
  H.g_w0 = h->P(L.gate.w0); H.g_b0 = h->P(L.gate.b0); H.g_w1 = h->P(L.gate.w1); H.g_b1 = h->P(L.gate.b1);
  H.t_w0 = h->P(L.tower.w0); H.t_b0 = h->P(L.tower.b0); H.t_w1 = h->P(L.tower.w1); H.t_b1 = h->P(L.tower.b1);
  H.t_wo = h->P(L.tower.wout); H.t_bo = h->P(L.tower.bout);
  H.ds_w0 = h->G(L.score.w0); H.ds_b0 = h->G(L.score.b0); H.ds_w1 = h->G(L.score.w1); H.ds_b1 = h->G(L.score.b1);
  H.de_w0 = h->G(L.expert.w0); H.de_b0 = h->G(L.expert.b0); H.de_w1 = h->G(L.expert.w1); H.de_b1 = h->G(L.expert.b1);
  H.dg_w0 = h->G(L.gate.w0); H.dg_b0 = h->G(L.gate.b0); H.dg_w1 = h->G(L.gate.w1); H.dg_b1 = h->G(L.gate.b1);
  H.dt_w0 = h->G(L.tower.w0); H.dt_b0 = h->G(L.tower.b0); H.dt_w1 = h->G(L.tower.w1); H.dt_b1 = h->G(L.tower.b1);
  H.dt_wo = h->G(L.tower.wout); H.dt_bo = h->G(L.tower.bout);
  H.wT = h->wf("head.wT");
  static_assert(kHead2Groups == 8, "layout.h: bn.gsums / bn.gbsums hold 8 copies");
  for (int i = 0; i < BN_COUNT; ++i) {
    H.bn[i] = h->bn[i];
    // set i's copies are contiguous: [kHead2Groups][C_i][2], sets one after the other
    H.gsums[i] = h->wd("bn.gsums") + (size_t)kHead2Groups * L.bn_bsums_off[i];
    H.gbsums[i] = h->wd("bn.gbsums") + (size_t)kHead2Groups * L.bn_bsums_off[i];
  }
  H.z1 = h->wf("z1"); H.z2 = h->wf("z2"); H.aw = h->wf("pool.aw"); H.new_long = h->wf("new_long");
  H.ze0 = h->wf("ze0"); H.zg0 = h->wf("zg0"); H.ze1 = h->wf("ze1"); H.zg1 = h->wf("zg1"); H.u = h->wf("u");
  H.zt0 = h->wf("zt0"); H.zt1 = h->wf("zt1"); H.logits = h->wf("logits");
  H.d_logits = h->wf("d_logits"); H.d_t1 = h->wf("d_t1"); H.d_t0 = h->wf("d_t0"); H.d_e1 = h->wf("d_e1"); H.d_g1 = h->wf("d_g1");
  H.d_e0 = h->wf("d_e0"); H.d_g0 = h->wf("d_g0"); H.d_new_long = h->wf("d_new_long"); H.d_tgt = h->wf("d_tgt");
  H.d_z2 = h->wf("d_z2"); H.g_a = h->wf("g_a");
  H.loss_acc = h->wd("loss_acc"); H.dp_scalars = h->wd("dp.scalars");
  const int g2 = head2_grid();
  if (g2 <= 0) { cudaGetLastError(); return 0; }           // no cooperative launch on this device: stand-alone kernels
  if (!h->head_bar) {
    if (cudaMalloc(&h->head_bar, 256 + 2 * 32 * 8) != cudaSuccess) return check_cuda(h, "head barrier alloc");
    cudaMemsetAsync(h->head_bar, 0, 256 + 2 * 32 * 8, st);
  }
  h->head2_grid = g2;
  return check_cuda(h, "head2");
}

// The stand-alone head's backward pass (kernels_head.cu), loss through attention pooling: the gradient of blk1.out ends in g_a, the
// weight-gradient GEMMs (no consumer before the optimiser) run on the side stream.  Data parallel: the batch-norm gradient sums are
// summed over the ranks by NCCL.  Returns non-zero when an NCCL call failed; the caller reports it after joining the side stream.
static int head_backward(PamrecHandle h, const PamrecBatch* b, cudaStream_t st) {
  const Layout& L = h->L;
  const int B = b->batch, T = h->cfg.max_seq_len;
  const int W = h->cfg.world_size;
  const int Bg = b->global_batch > 0 ? b->global_batch : B * W;
  const float gs = 1.0f / (float)W;    // BN parameter gradients are already global: the dense all-reduce sums W copies
  BnSet* bn = h->bn;
  int crc = 0;
  launch_loss(h->wf("logits"), b->labels_satisfied, b->labels_play, b->plays, h->wf("d_logits"), h->wd("loss_acc"), B, Bg,
              W > 1 ? h->wd("dp.scalars") : nullptr, h->cfg.fuzhu_weight, h->cfg.order_weight,
              h->cfg.loss_kind == PAMREC_LOSS_SOFTMAX ? h->cfg.softmax_group : 0, st);
  // Batch-norm backward is folded into the dense kernels (common.cuh: BnGrad / BnGradOut): the kernel that produces a
  // gradient buffer also accumulates the two column sums of its layer's BN, the consumers turn dA into dz while loading.
  // Buffers produced by the mixing / pooling kernels get their sums from k_bn_bwd_stats.  Data parallel: sums over ranks.
  cudaMemsetAsync(h->wd("bn.bsums"), 0, (size_t)L.ws[L.ws_index.at("bn.bsums")].numel * sizeof(double), st);
  auto sync_bsums = [&](const std::vector<int>& ids) {
    if (W == 1 || crc) return;
    PAMREC_PROF("allreduce_bn_bwd", 1, st);
    crc |= h->comm.group_start();
    for (int id : ids) crc |= h->comm.all_reduce(bn[id].bsums, 2 * (int64_t)bn[id].C, COMM_F64, st);
    crc |= h->comm.group_end();
  };
  const HeadMlps m = head_mlps(h, b);
  mlp_backward(h, {&m.tower}, gs, sync_bsums, st);
  launch_combine_bwd(h->wf("ze1"), h->wf("zg1"), bn[BN_E1], bn[BN_G1], h->wf("d_u"), h->wf("d_e1"), h->wf("d_g1"),
                     h->wf("d_tgt"), B, st);
  mlp_backward(h, {&m.expert, &m.gate}, gs, sync_bsums, st);
  // ---- attention pooling
  launch_pool_bwd(h->wf("blk1.out"), h->wf("z2"), bn[BN_S1], b->mask, h->wf("d_new_long"), h->wf("d_z2"), h->wf("g_a"), B, T, st);
  mlp_backward(h, {&m.score}, gs, sync_bsums, st);
  return crc;
}

int pamrec_backward(PamrecHandle h, const PamrecBatch* b, void* stream) {
  if (int rc = check_batch(h, b, true)) return rc;
  ProfBind _pb(h);
  cudaStream_t st = (cudaStream_t)stream;
  if (h->cfg.model_kind == PAMREC_MODEL_SASREC) return sas_backward(h, b, st);
  if (h->sibling()) return sib_backward(h, b, st);
  const Layout& L = h->L;
  const int B = b->batch, T = h->cfg.max_seq_len, N = B * T;
  int crc = 0;
  cudaMemsetAsync(h->buf.dense_grad, 0, (size_t)L.dense_numel * 4, st);
  cudaMemsetAsync(h->wd("loss_acc"), 0, 8 * sizeof(double), st);
  cudaMemsetAsync(h->wd("sp_normsq"), 0, 8 * sizeof(double), st);
  if (h->use_head2()) {
    cudaMemsetAsync(h->wd("bn.bsums"), 0, (size_t)L.ws[L.ws_index.at("bn.bsums")].numel * sizeof(double), st);
    // loss + the dX chain of the head as ONE persistent cooperative kernel; the weight gradients (no consumer before the
    // optimiser) run on the side stream beside the encoder's backward pass
    HeadDyn d = head_dyn(h, b, true, 12);
    if (launch_head2_bwd(h->head2, d, h->head2_grid, st)) return check_cuda(h, "cooperative head launch");
    h->fork(st, [&](cudaStream_t s2) { launch_head2_dw(h->head2, B, s2); });
  } else {
    crc = head_backward(h, b, st);
  }
  float* g_a = h->wf("g_a");
  float* g_b = h->wf("g_b");
  // ---- encoder blocks (grad of blk1.out is in g_a)
  const int max_tiles = N / kTokTile + kNB + 1;
  int* ctl = h->wi("bucket_ctl");
  for (int k = 1; k >= 0; --k) {
    const BlockOff& o = L.blk[k];
    std::string p = "blk" + std::to_string(k) + ".";
    const float* xin = k == 0 ? h->wf("x0") : h->wf("blk0.out");
    float* gout = k == 1 ? g_a : g_b;
    float* gin = k == 1 ? g_b : g_a;
    // block 1's weight-gradient inputs must outlive block 0's backward, which rewrites d_Q / d_K / d_V and g_a (layout.h)
    float* dQ = h->wf(k == 1 ? "blk1.d_Q" : "d_Q");
    float* dK = h->wf(k == 1 ? "blk1.d_K" : "d_K");
    float* dV = h->wf(k == 1 ? "blk1.d_V" : "d_V");
    float* dout = k == 1 ? h->wf("blk1.d_out") : gout;
    // the block's weight gradients (no consumer before the optimiser) run on the side stream, each half as soon as its inputs
    // exist: the FFN pair after the FFN backward, the projection after the attention backward; joined at the end of the pass
    EncDwArgs dw{h->wf(p + "qin"), xin, dQ, dK, dV, h->wi("perm"), ctl, h->wf(p + "y"), h->P(o.ln_b_beta), h->P(o.ln_b_gamma),
                 h->wf(p + "h"), h->wf(p + "dhr"), dout, h->G(o.wq), h->G(o.wk), h->G(o.wv), h->G(o.w1), h->G(o.b1), h->G(o.w2),
                 h->G(o.b2), N, true};
    launch_ffn_bwd(h->wf(p + "y"), gout, h->P(o.w1), h->P(o.b1), h->P(o.w2), h->P(o.ln_b_beta), h->P(o.ln_b_gamma), h->wf("d_y"),
                   h->wf(p + "h"), h->wf(p + "dhr"), k == 1 ? dout : nullptr, h->G(o.ln_b_beta), h->G(o.ln_b_gamma), N, st);
    h->fork(st, [&](cudaStream_t s2) { launch_enc_dw(dw, s2); });
    // backward: the MMA kernel keeps K, V, Q and dY of a sample in shared memory (141 KB at T = 200: one CTA per SM), measured slower
    // than the FFMA kernel there (8.5 vs 6.4 ms per step on long_b4095_t200) and faster below (T = 100: 230 vs 292 us, T = 50: 152 vs 196 us)
    if (T <= 128)
      launch_attn_bwd_mma(h->wf(p + "Q"), h->wf(p + "K"), h->wf(p + "V"), h->wf("d_y"), h->wf(p + "pv"), h->wf(p + "ml"),
                          b->mask, dQ, dK, dV, B, T, st);
    else
      launch_attn_bwd(h->wf(p + "Q"), h->wf(p + "K"), h->wf(p + "V"), h->wf("d_y"), h->wf(p + "pv"), h->wf(p + "ml"),
                      b->mask, dQ, dK, dV, B, T, st);
    dw.ffn = false;
    h->fork(st, [&](cudaStream_t s2) { launch_enc_dw(dw, s2); });
    launch_proj_bwd(xin, h->wf("d_y"), dQ, dK, dV, h->wi("perm"), ctl, h->wi("tile_bucket"), h->wi("tile_begin"), h->wi("tile_count"),
                    max_tiles, h->P(o.wq), h->P(o.wk), h->P(o.wv), h->P(o.ln_a_beta), h->P(o.ln_a_gamma), gin, h->G(o.ln_a_beta),
                    h->G(o.ln_a_gamma), st);
  }
  // dX0 is in g_a
  launch_embed_bwd_reduce(g_a, h->wf("d_tgt"), h->wf("d_tgt_total"), h->G(L.pos), h->wd("sp_normsq") + 4,
                          h->sharded() ? nullptr : h->wd("sp_normsq"), B, T, st);
  h->join(st);                    // the head's and the encoder's weight gradients (side stream) are complete from here on
  if (crc) return fail(h, "nccl: %s", h->comm.err.c_str());
  return check_cuda(h, "backward");
}

// dense gradients (+ the replicated tables' gradient tables, already in the exchange buffer), clip norms and loss sums summed
// over the ranks through peer memory (kernels_p2p.cu:k_xr_*)
static void peer_allreduce_grads(PamrecHandle h, cudaStream_t st) {
  XrArgs a;
  memset(&a, 0, sizeof a);
  const int W = h->cfg.world_size;
  for (int p = 0; p < W; ++p) a.peer[p] = h->xr_region(p);
  a.world = W; a.rank = h->cfg.rank; a.epoch = ++h->xr_epoch;
  a.cap = p2p_xr_cap(W, h->xr_floats());
  a.dense_grad = h->buf.dense_grad; a.n_dense = h->L.dense_numel;
  a.scalars[0] = h->wd("sp_normsq"); a.n_scalars[0] = 8;
  a.scalars[1] = h->wd("loss_acc"); a.n_scalars[1] = 4;
  a.counter = reinterpret_cast<unsigned*>(h->xr_region(h->cfg.rank) + 128);
  a.err = h->mbox_err();
  launch_xr_allreduce(a, h->buf.dense_grad, st);
}

// ------------------------------------------------------------------------------------------
int pamrec_apply_gradients(PamrecHandle h, const PamrecBatch* b, int64_t step, void* stream) {
  if (int rc = check_batch(h, b, true)) return rc;
  ProfBind _pb(h);
  // step >= 1: the caller counts the steps; step == 0: the device counter advances by one ("adam.step", for a step replayed from
  // a CUDA graph: a host-computed step size would be frozen into the graph).  Whole-table layouts only.
  if (h->sibling()) return sib_apply(h, b, step, (cudaStream_t)stream);
  if (step < 0) return fail(h, "step must be >= 1 (or 0: advance the device step counter)");
  if (step == 0 && (h->sharded() || h->cfg.world_size > 1)) return fail(h, "the device step counter (step = 0) needs one GPU with whole tables");
  cudaStream_t st = (cudaStream_t)stream;
  const Layout& L = h->L;
  const PamrecConfig& c = h->cfg;
  const int B = b->batch, T = c.max_seq_len;
  const double b1 = c.beta1, b2 = c.beta2;
  const double tstep = step > 0 ? (double)step : 1.0;
  const float lr_t = (float)((double)c.learning_rate * std::sqrt(1.0 - std::pow(b2, tstep)) / (1.0 - std::pow(b1, tstep)));
  const float* lr_dev = nullptr;
  if (!h->sharded()) {
    // whole tables: every Adam kernel of this step reads lr_t from the device
    launch_adam_step(step, h->wd("adam.step"), c.learning_rate, c.beta1, c.beta2, h->wf("adam.lr"), st);
    lr_dev = h->wf("adam.lr");
  }
  double* reg = h->wd("loss_acc") + 3;
  void* tmp = h->ws<char>("cub_temp");
  size_t tmp_bytes = (size_t)L.ws[L.ws_index.at("cub_temp")].numel;
  bool dense_aside = false;
  const float* dX0 = h->wf("g_a");
  const float* dT = h->wf("d_tgt_total");
  if (h->sharded()) {
    // ---- row-sharded tables: local pre-reduction, row gradients to their owners, owner-side merge + Adam
    Comm& cm = h->comm;
    int crc = 0;
    if (!h->xc_users) return fail(h, "apply_gradients needs pamrec_forward(training=1) on the same batch");   // before any collective
    for (const IdTables& s : h->sp) {
      if (!s.d->accum) continue;
      const GradRows g{dX0, kD, dT, kE, s.d->col};
      if (int rc = sparse_reduce(h, s.req, s.d->lookups(B, T), s.d->n_hist(B, T), &g, nullptr, 0, st)) return rc;
    }
    {
      PAMREC_PROF("xchg_grads", 1, st);
      crc |= cm.group_start();
      for (const IdTables& s : h->sp)
        if (s.d->accum)
          crc |= cm.all_to_all_v(s.req.accum, s.x.soff.data(), s.x.scnt.data(), s.xrows, s.x.roff.data(), s.x.rcnt.data(), s.d->width,
                                 COMM_F32, st);
      crc |= cm.group_end();
    }
    cudaStreamWaitEvent(st, h->ev_plan, 0);            // owner-side plans (side stream, forked in the forward exchange)
    for (const IdTables& s : h->sp) {
      const GradRows g{s.xrows, s.d->width, nullptr, 0, 0};
      if (int rc = sparse_reduce(h, s.own, s.x.n_recv, s.x.n_recv, s.d->accum ? &g : nullptr, s.tab, s.d->n_tab, st)) return rc;
    }
    if (h->use_xr()) {
      peer_allreduce_grads(h, st);
    } else {
      PAMREC_PROF("allreduce_grads", 1, st);
      crc |= cm.group_start();
      crc |= cm.all_reduce(h->buf.dense_grad, L.dense_numel, COMM_F32, st);
      crc |= cm.all_reduce(h->wd("sp_normsq"), 8, COMM_F64, st);
      crc |= cm.all_reduce(h->wd("loss_acc"), 4, COMM_F64, st);     // data, aux, order, embedding part of the L2 term
      crc |= cm.group_end();
    }
    if (crc) return fail(h, "nccl: %s", cm.err.c_str());
    for (const IdTables& s : h->sp)
      if (int rc = sparse_apply(h, s.tab, s.d->n_tab, s.x.n_recv, lr_t, st)) return rc;
  } else {
    // ---- whole tables on this GPU: one-sort plan (side stream, beside the forward pass) -> run walk -> Adam
    if (c.world_size == 1) {
      // one GPU: the dense variables' clip norms + Adam share nothing with the tables' walk + sweep: side stream, joined before the losses
      dense_aside = true;
      h->fork(st, [&](cudaStream_t s2) {
        launch_dense_norm(h->buf.dense_param, h->buf.dense_grad, h->wi("seg_tab"), (int)L.dense.size(), c.layer_l2, h->wd("seg_normsq"),
                          h->wd("sp_normsq") + 4, reg, s2);
        launch_dense_adam(h->buf.dense_param, h->buf.dense_grad, h->buf.dense_m, h->buf.dense_v, h->wi("seg_id"), h->wi("seg_tab"),
                          h->wd("seg_normsq"), L.dense_numel, c.layer_l2, lr_t, lr_dev, c.beta1, c.beta2, c.epsilon, c.max_grad_norm,
                          c.is_clip_norm, s2);
      });
    }
    const bool planned = h->plan_for == b->item_history && h->plan_rows == B;
    h->plan_for = nullptr;
    const Sp2 s2 = make_sp2(h, b);
    AdamP ap = make_adam(h, lr_t);
    ap.lr_dev = lr_dev;
    if (planned) cudaStreamWaitEvent(st, h->ev_plan, 0);
    else if (launch_sp2_plan(s2, tmp, tmp_bytes, st)) return fail(h, "cub sort failed");
    launch_sp2_walk(s2, ap, st);
   
    if (h->replicated()) {
      // replicated tables: gradient tables + touch counts, dense gradients, clip norms and losses summed over the ranks
      Sp2 s3 = s2;                                           // after the all-reduce: the summed gradient tables
      if (h->use_xr()) {
        peer_allreduce_grads(h, st);
        s3.rep_grad = h->rep_grad_out();
      } else {
        Comm& cm = h->comm;
        int crc = 0;
        {
          PAMREC_PROF("allreduce_grads", 1, st);
          crc |= cm.group_start();
          crc |= cm.all_reduce(h->buf.dense_grad, L.dense_numel, COMM_F32, st);
          crc |= cm.all_reduce(s2.rep_grad, sp2_rep_floats(c.n_items, c.n_cates, c.n_users), COMM_F32, st);
          crc |= cm.all_reduce(h->wd("sp_normsq"), 8, COMM_F64, st);
          crc |= cm.all_reduce(h->wd("loss_acc"), 4, COMM_F64, st);
          crc |= cm.group_end();
        }
        if (crc) return fail(h, "nccl: %s", cm.err.c_str());
      }
      launch_sp2_rep_l2(s3, st);
      launch_sp2_adam_sweep(s3, ap, c.sparse_adam_mode == PAMREC_ADAM_LAZY ? 1 : 0, st);
     
    } else if (s2.mode == SP2_FUSED) {
      launch_sp2_lazy_finish(s2, ap, st);
    } else {
      launch_sp2_adam_sweep(s2, ap, 0, st);
    }
  }
  const int n_seg = (int)L.dense.size();
  if (dense_aside) {
    h->join(st);
  } else {
    launch_dense_norm(h->buf.dense_param, h->buf.dense_grad, h->wi("seg_tab"), n_seg, c.layer_l2, h->wd("seg_normsq"),
                      h->wd("sp_normsq") + 4, reg, st);
    launch_dense_adam(h->buf.dense_param, h->buf.dense_grad, h->buf.dense_m, h->buf.dense_v, h->wi("seg_id"), h->wi("seg_tab"),
                      h->wd("seg_normsq"), L.dense_numel, c.layer_l2, lr_t, lr_dev, c.beta1, c.beta2, c.epsilon, c.max_grad_norm,
                      c.is_clip_norm, st);
  }
  launch_finish_losses(h->wd("loss_acc"), h->wf("losses"), h->sharded() ? nullptr : h->wd("sp2.l2sq"), c.embed_l2, h->wd("sp_normsq"), st);
 
  return check_cuda(h, "apply_gradients");
}

#include "api_sibling.inl"
#include "api_rank.inl"
#include "api_attn.inl"

int pamrec_train_step(PamrecHandle h, const PamrecBatch* b, int64_t step, float* losses_out, void* stream) {
  if (!h) return -1;
  const int64_t l0 = h->prof.launches;
  if (int rc = pamrec_forward(h, b, 1, nullptr, stream)) return rc;
  if (int rc = pamrec_backward(h, b, stream)) return rc;
  if (int rc = pamrec_apply_gradients(h, b, step, stream)) return rc;
  if (losses_out)
    cudaMemcpyAsync(losses_out, h->wf("losses"), 5 * sizeof(float), cudaMemcpyDeviceToDevice, (cudaStream_t)stream);
  h->launches = h->prof.launches - l0;
  return check_cuda(h, "train_step");
}

int pamrec_comm_all_reduce(PamrecHandle h, void* dptr, int64_t count, int dtype, void* stream) {
  if (!h) return -1;
  CommType t = dtype == PAMREC_F64 ? COMM_F64 : (dtype == PAMREC_I32 ? COMM_I32 : COMM_F32);
  if (h->comm.all_reduce(dptr, count, t, (cudaStream_t)stream)) return fail(h, "nccl: %s", h->comm.err.c_str());
  return 0;
}

int pamrec_histograms(PamrecHandle h, const float* const* ptrs, const int64_t* counts, int n, int reduce, const int64_t* out_offsets,
                      double* stats, double* out, void* scratch, int64_t* scratch_bytes, void* stream) {
  if (!h) return -1;
  if (n < 1 || n > kHistMaxSeg || !counts || !scratch_bytes) return fail(h, "histograms: 1 to %d segments and their counts", kHistMaxSeg);
  const double* pos = hist_positive_limits();
  if (!pos) return fail(h, "histograms: the default bucket table does not have %d positive limits", kHistPos);
  static thread_local HistArgs a;                          // ~20 KB: not on the stack
  std::copy(pos, pos + kHistPos, a.pos);
  a.n = n; a.world = h->cfg.world_size; a.rank = h->cfg.rank;
  int64_t items = 0;
  for (int s = 0; s < n; ++s) {
    if (counts[s] < 0 || counts[s] >= ((int64_t)1 << 31)) return fail(h, "histograms: segment %d has %lld elements", s, (long long)counts[s]);
    a.first_item[s] = (int)items;
    items += hist_items(counts[s]);
  }
  if (items >= ((int64_t)1 << 31)) return fail(h, "histograms: too many elements");
  a.first_item[n] = (int)items;
  const size_t bins_bytes = ((size_t)n * kHistBuckets * sizeof(int) + 255) / 256 * 256;
  const int64_t need = (int64_t)(bins_bytes + (size_t)items * 5 * sizeof(double));
  if (!scratch) { *scratch_bytes = need; return 0; }
  if (*scratch_bytes < need) return fail(h, "histograms: scratch of %lld bytes, %lld needed", (long long)*scratch_bytes, (long long)need);
  if (!ptrs || !out_offsets || !stats || !out) return fail(h, "histograms: null argument");
  for (int s = 0; s <= n; ++s) {
    a.out_off[s] = out_offsets[s];
    if (s < n && (out_offsets[s + 1] < out_offsets[s] || (counts[s] && !ptrs[s]))) return fail(h, "histograms: segment %d", s);
  }
  for (int s = 0; s < n; ++s) { a.ptr[s] = ptrs[s]; a.count[s] = counts[s]; }
  ProfBind _pb(h);
  cudaStream_t st = (cudaStream_t)stream;
  int* bins = static_cast<int*>(scratch);
  double* part = reinterpret_cast<double*>(static_cast<char*>(scratch) + bins_bytes);
  cudaMemsetAsync(bins, 0, (size_t)n * kHistBuckets * sizeof(int), st);
  launch_hist_bin(a, (int)items, bins, part, stats, st);
  if (reduce && a.world > 1) {
    if (h->comm.all_reduce(bins, (int64_t)n * kHistBuckets, COMM_I32, st) ||
        h->comm.all_reduce(stats, (int64_t)n * hist_stats_width(a.world), COMM_F64, st))
      return fail(h, "nccl: %s", h->comm.err.c_str());
  }
  launch_hist_compact(a, bins, stats, out, st);
  return check_cuda(h, "histograms");
}

int pamrec_histogram_buckets(const int32_t* counts, double* limits_out, double* pairs_out, int* n_pairs) {
  const double* pos = hist_positive_limits();
  if (!pos) return -1;
  if (limits_out)
    for (int b = 0; b < kHistBuckets; ++b) limits_out[b] = hist_limit(pos, b);
  if (counts) {
    if (!pairs_out || !n_pairs) return -1;
    int k = 0;
    for (int b = 0; b < kHistBuckets; ++b)
      if (hist_emits(counts, b)) { pairs_out[2 * k] = hist_limit(pos, b); pairs_out[2 * k + 1] = (double)counts[b]; ++k; }
    *n_pairs = k;
  }
  return 0;
}

int pamrec_bench_gather(PamrecHandle h, const int32_t* item_ids, const int32_t* cate_ids, const int32_t* tgt_items,
                        const int32_t* tgt_cates, int64_t n_rows, int32_t T, float* out, void* stream) {
  if (!h || !h->bound) return fail(h, "not bound");
  if (h->sibling()) return fail(h, "bench_gather measures PAMRec's fused gather");
  if (T < 1 || T > h->cfg.max_seq_len) return fail(h, "T outside the position table");
  ProfBind _pb(h);
  launch_embed_fwd(item_ids, cate_ids, tgt_items, tgt_cates, h->buf.item_w, h->buf.cate_w, h->P(h->L.pos), out, nullptr, n_rows,
                   T, (cudaStream_t)stream);
  return check_cuda(h, "bench_gather");
}

int pamrec_bench_table_adam(PamrecHandle h, int64_t step, void* stream) {
  if (!h || !h->bound) return fail(h, "not bound");
  ProfBind _pb(h);
  const PamrecConfig& c = h->cfg;
  const double b1 = c.beta1, b2 = c.beta2;
  const float lr_t = (float)((double)c.learning_rate * std::sqrt(1.0 - std::pow(b2, (double)step)) / (1.0 - std::pow(b1, (double)step)));
  if (h->sharded() || h->sibling()) return fail(h, "bench_table_adam runs on PAMRec's whole tables");
  PamrecBatch nb;
  memset(&nb, 0, sizeof nb);
  Sp2 s2 = make_sp2(h, &nb);                              // no lookups: every row decays, none is touched
  s2.mode = SP2_COMPACT; s2.slot = h->wi("sp2.slot");
  launch_sp2_adam_sweep(s2, make_adam(h, lr_t), 0, (cudaStream_t)stream);
  return check_cuda(h, "bench_table_adam");
}

int pamrec_set_debug(PamrecHandle h, int flags) {
  if (!h) return -1;
  h->debug = flags;
  h->head_trace = (flags & PAMREC_DEBUG_HEAD_TRACE) != 0;
  if (h->head_trace && !h->head_trace_cta && cudaMalloc(&h->head_trace_cta, 2 * 16 * 256 * 8) == cudaSuccess)
    cudaMemset(h->head_trace_cta, 0, 2 * 16 * 256 * 8);
  return 0;
}
int pamrec_head_trace_ctas(PamrecHandle h, int backward, uint64_t* out /* [16][256] */) {
  if (!h || !out || !h->head_trace_cta) return -1;
  cudaDeviceSynchronize();
  if (cudaMemcpy(out, h->head_trace_cta + (backward ? 16 * 256 : 0), 16 * 256 * 8, cudaMemcpyDeviceToHost) != cudaSuccess) return check_cuda(h, "head trace");
  return 0;
}
int pamrec_head_trace(PamrecHandle h, int backward, uint64_t out[32]) {
  if (!h || !out || !h->head_bar) return -1;
  cudaDeviceSynchronize();
  if (cudaMemcpy(out, reinterpret_cast<unsigned long long*>(h->head_bar + 64) + (backward ? 32 : 0), 32 * 8, cudaMemcpyDeviceToHost) != cudaSuccess)
    return check_cuda(h, "head trace");
  return 0;
}
int pamrec_profile_enable(PamrecHandle h, int on) {
  if (!h) return -1;
  h->prof.on = on != 0;
  return 0;
}
int pamrec_profile_reset(PamrecHandle h) {
  if (!h) return -1;
  h->prof.reset();
  return 0;
}
int pamrec_profile_count(PamrecHandle h) {
  if (!h) return -1;
  h->prof.resolve();
  return (int)h->prof.names.size();
}
int pamrec_profile_get(PamrecHandle h, int index, char name[64], double* total_ms, int64_t* launches) {
  if (!h || index < 0 || index >= (int)h->prof.names.size()) return -1;
  snprintf(name, 64, "%s", h->prof.names[index].c_str());
  if (total_ms) *total_ms = h->prof.ms[index];
  if (launches) *launches = h->prof.cnt[index];
  return 0;
}

}  // extern "C"
