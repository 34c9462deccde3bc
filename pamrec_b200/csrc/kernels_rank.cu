// Candidate ranking (pamrec_rank_candidates, api_rank.inl): the candidate map, the expansion of lines x candidates into scoring
// rows, SASRec's tower input, and the streaming top-K merge.  Order everywhere: score descending, then item id ascending.
#include <cmath>

#include "kernels.h"

namespace pamrec {

// a is ordered before b
__device__ __forceinline__ bool rank_before(float sa, int ia, float sb, int ib) { return sa > sb || (sa == sb && ia < ib); }

// map[item] = candidate index; flags[0] = 1 + a candidate whose id is outside [1, n_items), flags[1] = 1 + a duplicate,
// flags[2] = 1 + a candidate whose category is outside [0, n_cates)
__global__ void k_rank_map(const int* __restrict__ items, const int* __restrict__ cates, int n, int n_items, int n_cates, int* map,
                           int* flags) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n) return;
  const int id = items[c], ct = cates[c];
  if (id < 1 || id >= n_items) { atomicCAS(flags + 0, 0, c + 1); return; }
  if (ct < 0 || ct >= n_cates) { atomicCAS(flags + 2, 0, c + 1); return; }
  if (atomicCAS(map + id, -1, c) != -1) atomicCAS(flags + 1, 0, c + 1);
}
void launch_rank_map(const int* items, const int* cates, int n, int n_items, int n_cates, int* map, int* flags, cudaStream_t st) {
  PAMREC_PROF("rank_map", 1, st);
  k_rank_map<<<(n + 255) / 256, 256, 0, st>>>(items, cates, n, n_items, n_cates, map, flags);
}

// Per line: the row that scores its own item (the candidate's category when the item is a candidate), a zero rank count, and an
// empty top K (id -1, score -inf).
__global__ void k_rank_begin(const int* __restrict__ items, const int* __restrict__ cates, const int* __restrict__ map,
                             const int* __restrict__ cand_cates, int n_items, int B, int K, int* own_items, int* own_cates, int* count,
                             int* topk_items, float* topk_scores) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (int64_t)B * K) { topk_items[i] = -1; topk_scores[i] = -INFINITY; }
  if (i < B) {
    const int id = items[i];
    const int c = id >= 0 && id < n_items ? map[id] : -1;
    own_items[i] = id;
    own_cates[i] = c >= 0 ? cand_cates[c] : cates[i];
    count[i] = 0;
  }
}
void launch_rank_begin(const int* items, const int* cates, const int* map, const int* cand_cates, int n_items, int B, int K,
                       int* own_items, int* own_cates, int* count, int* topk_items, float* topk_scores, cudaStream_t st) {
  PAMREC_PROF("rank_begin", 1, st);
  const int64_t n = (int64_t)B * K;
  k_rank_begin<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(items, cates, map, cand_cates, n_items, B, K, own_items, own_cates, count,
                                                            topk_items, topk_scores);
}

// Rows p0 .. p0 + rows - 1 of the line-major pairs (line = p / n_cand, candidate = p % n_cand): the line's history arrays, its
// user, and the candidate as the target.  One thread per (row, position).
__global__ void k_rank_expand(const RankRows a, RankBatch d, int64_t p0, int rows, int n_cand, int T) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)rows * T) return;
  const int r = (int)(i / T), t = (int)(i % T);
  const int64_t p = p0 + r;
  const int64_t l = p / n_cand;
  const int64_t s = l * T + t;
  d.item_history[i] = a.item_history[s];
  d.cate_history[i] = a.cate_history[s];
  d.mask[i] = a.mask[s];
  if (a.loop_times) d.loop_times[i] = a.loop_times[s];
  if (a.sat_item) { d.sat_item[i] = a.sat_item[s]; d.sat_cate[i] = a.sat_cate[s]; d.sat_mask[i] = a.sat_mask[s]; }
  if (t == 0) {
    const int c = (int)(p - l * n_cand);
    d.items[r] = a.cand_items[c];
    d.cates[r] = a.cand_cates[c];
    if (a.users) d.users[r] = a.users[l];
  }
}
void launch_rank_expand(const RankRows& a, const RankBatch& d, int64_t p0, int rows, int n_cand, int T, cudaStream_t st) {
  PAMREC_PROF("rank_expand", 1, st);
  const int64_t n = (int64_t)rows * T;
  k_rank_expand<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a, d, p0, rows, n_cand, T);
}

// SASRec's tower input of rows p0 .. p0 + rows - 1: U[r] = final state of the line (U_lines[l, 0:S]) | item_w[c] | cate_w[cate(c)],
// the row sas_final_fwd builds for that line with the candidate as its target.
__global__ void k_rank_tower_in(const float* __restrict__ U_lines, const int* __restrict__ cand_items, const int* __restrict__ cand_cates,
                                const float* __restrict__ item_w, const float* __restrict__ cate_w, float* __restrict__ U, int64_t p0,
                                int rows, int n_cand, int I, int Cw) {
  const int S = I + Cw;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)rows * 2 * S) return;
  const int r = (int)(i / (2 * S)), j = (int)(i % (2 * S));
  const int64_t p = p0 + r;
  const int64_t l = p / n_cand;
  const int c = (int)(p - l * n_cand);
  float v;
  if (j < S) v = U_lines[l * 2 * S + j];
  else if (j < S + I) v = item_w[(int64_t)cand_items[c] * I + (j - S)];
  else v = cate_w[(int64_t)cand_cates[c] * Cw + (j - S - I)];
  U[i] = v;
}
void launch_rank_tower_in(const float* U_lines, const int* cand_items, const int* cand_cates, const float* item_w, const float* cate_w,
                          float* U, int64_t p0, int rows, int n_cand, int item_dim, int cate_dim, cudaStream_t st) {
  PAMREC_PROF("rank_tower_in", 1, st);
  const int64_t n = (int64_t)rows * 2 * (item_dim + cate_dim);
  k_rank_tower_in<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(U_lines, cand_items, cand_cates, item_w, cate_w, U, p0, rows, n_cand,
                                                               item_dim, cate_dim);
}

// Streaming top-K merge, one CTA per line that rows p0 .. p0 + rows - 1 touch.  The line's running top K and a tile of its new
// candidates (excluded ones and the tail as sentinels: id -1, score -inf) are sorted together in shared memory by a bitonic
// sort of up to kRankSortN entries; the first K stay.  Candidates ordered before the line's own item are counted for its rank.  A
// non-finite score records 1 + the line in flags[3] and is left out.
constexpr int kRankSortN = 2048;
constexpr int kRankThreads = 1024;
__global__ void __launch_bounds__(kRankThreads) k_rank_merge(RankMerge a) {
  __shared__ float s_sc[kRankSortN];
  __shared__ int s_id[kRankSortN];
  __shared__ int s_hist[PAMREC_MAX_T];
  __shared__ int s_cnt;
  const int tid = threadIdx.x;
  const int64_t l = a.l0 + blockIdx.x;
  const int64_t base = l * a.n_cand - a.p0;                       // row of candidate c: base + c
  const int c_begin = (int)(base < 0 ? -base : 0);
  const int c_end = (int)min((int64_t)a.n_cand, (int64_t)a.rows - base);
  const int K = a.K, T = a.T;
  for (int t = tid; t < T; t += kRankThreads)
    s_hist[t] = a.exclude && a.mask[l * T + t] > 0 ? a.item_history[l * T + t] : -1;
  for (int i = tid; i < K; i += kRankThreads) { s_sc[i] = a.topk_scores[l * K + i]; s_id[i] = a.topk_items[l * K + i]; }
  if (tid == 0) s_cnt = 0;
  const int own = a.own_items[l];
  const float own_s = a.own_scores[l];
  const bool own_valid = own >= 0 && own < a.n_items && a.map[own] >= 0;
  int cnt = 0;
  int N = kRankSortN;                                              // the smallest power of two that takes K + the whole segment
  while (N > 64 && N / 2 >= K + (c_end - c_begin)) N >>= 1;
  const int tile = N - K;
  __syncthreads();
  for (int c0 = c_begin; c0 < c_end; c0 += tile) {
    for (int i = tid; i < tile; i += kRankThreads) {
      const int c = c0 + i;
      float sc = -INFINITY;
      int id = -1;
      if (c < c_end) {
        const float v = a.scores[base + c];
        const int it = a.cand_items[c];
        bool keep = true;
        if (!isfinite(v)) { atomicCAS(a.flags + 3, 0, (int)l + 1); keep = false; }
        if (keep && a.exclude && it != own)
          for (int t = 0; t < T; ++t) keep &= s_hist[t] != it;
        if (keep) {
          sc = v; id = it;
          if (own_valid && it != own && rank_before(v, it, own_s, own)) ++cnt;
        }
      }
      s_sc[K + i] = sc; s_id[K + i] = id;
    }
    __syncthreads();
    for (int k = 2; k <= N; k <<= 1)
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int i = tid; i < N; i += kRankThreads) {
          const int p = i ^ j;
          if (p <= i) continue;
          const float si = s_sc[i], sp = s_sc[p];
          const int ii = s_id[i], ip = s_id[p];
          const bool first_half = (i & k) == 0;                    // this run sorts in rank order, the other in reverse
          if (first_half ? rank_before(sp, ip, si, ii) : rank_before(si, ii, sp, ip)) {
            s_sc[i] = sp; s_sc[p] = si; s_id[i] = ip; s_id[p] = ii;
          }
        }
        __syncthreads();
      }
  }
  atomicAdd(&s_cnt, cnt);
  __syncthreads();
  for (int i = tid; i < K; i += kRankThreads) { a.topk_scores[l * K + i] = s_sc[i]; a.topk_items[l * K + i] = s_id[i]; }
  if (tid == 0) a.count[l] += s_cnt;
}
void launch_rank_merge(const RankMerge& a, int n_lines, cudaStream_t st) {
  PAMREC_PROF("rank_merge", 1, st);
  k_rank_merge<<<n_lines, kRankThreads, 0, st>>>(a);
}

// own_rank[l] = 1 + count[l] when the line's item is a candidate, else -1; a non-finite score of the own item sets flags[3]
__global__ void k_rank_finish(const int* __restrict__ own_items, const float* __restrict__ own_scores, const int* __restrict__ map,
                              const int* __restrict__ count, int n_items, int B, int* own_rank, int* flags) {
  const int l = blockIdx.x * blockDim.x + threadIdx.x;
  if (l >= B) return;
  const int own = own_items[l];
  const bool valid = own >= 0 && own < n_items && map[own] >= 0;
  if (valid && !isfinite(own_scores[l])) atomicCAS(flags + 3, 0, l + 1);
  if (own_rank) own_rank[l] = valid ? 1 + count[l] : -1;
}
void launch_rank_finish(const int* own_items, const float* own_scores, const int* map, const int* count, int n_items, int B, int* own_rank,
                        int* flags, cudaStream_t st) {
  PAMREC_PROF("rank_finish", 1, st);
  k_rank_finish<<<(B + 255) / 256, 256, 0, st>>>(own_items, own_scores, map, count, n_items, B, own_rank, flags);
}

}  // namespace pamrec
