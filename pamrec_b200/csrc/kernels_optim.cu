// Sparse embedding backward (sorted ids -> warp-level segmented reduction -> row-wise Adam)
// and the dense-parameter optimiser.
//
// TF semantics reproduced (SURVEY.md section 7, H2 / H5):
//  * the gradient of an embedding table is the CONCATENATION of every lookup's rows
//    (history, target, and the L2 rows of tf.unique(ids)); tf.clip_by_norm (base_model.py:297-303)
//    takes its norm over those un-deduplicated rows;
//  * tf.train.AdamOptimizer then sums duplicate rows and, for sparse variables, decays m and v
//    and moves the weights of EVERY row of the table (mode DENSE_EXACT).  Mode LAZY touches
//    only the looked-up rows.
#include <cub/cub.cuh>

#include <climits>

#include "kernels.h"

namespace pamrec {

// ------------------------------------------------------------------------------------------
// d_tgt_total[b,:] = d_tgt_head[b,:] + sum_t dX0[b,t,20:40];  pos_normsq += |dX0|^2;
// dPos[t,:] += sum_b dX0[b,t,:]
__global__ void __launch_bounds__(128) k_dtgt_total(const float* __restrict__ dX0, const float* __restrict__ dTgtHead,
                                                    float* __restrict__ dTgtTotal, double* __restrict__ pos_normsq,
                                                    double* __restrict__ undedup, int T) {
  __shared__ double sh[3][4];
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* base = dX0 + (int64_t)b * T * kD;
  // squared norms of the rows this sample contributes to the three IndexedSlices gradients: position rows (all 40 columns),
  // item history rows (columns 0:16), category history rows (16:20); the target rows follow below
  double sq = 0.0, sq_i = 0.0, sq_c = 0.0;
  for (int i = tid; i < T * kD; i += 128) {
    const float v = base[i];
    const double q = (double)v * (double)v;
    const int col = i % kD;
    sq += q;
    if (col < kI) sq_i += q; else if (col < kE) sq_c += q;
  }
  if (tid < kE) {
    float s = dTgtHead[(int64_t)b * kE + tid];
    for (int t = 0; t < T; ++t) s += base[t * kD + kE + tid];
    dTgtTotal[(int64_t)b * kE + tid] = s;
    if (tid < kI) sq_i += (double)s * (double)s; else sq_c += (double)s * (double)s;
  }
  sq = warp_sum_d(sq); sq_i = warp_sum_d(sq_i); sq_c = warp_sum_d(sq_c);
  if ((tid & 31) == 0) { sh[0][tid >> 5] = sq; sh[1][tid >> 5] = sq_i; sh[2][tid >> 5] = sq_c; }
  __syncthreads();
  if (tid == 0) atomicAdd(pos_normsq, sh[0][0] + sh[0][1] + sh[0][2] + sh[0][3]);
  if (undedup != nullptr && (tid == 1 || tid == 2)) atomicAdd(undedup + (tid - 1), sh[tid][0] + sh[tid][1] + sh[tid][2] + sh[tid][3]);
}
constexpr int kPosRows = 64;
__global__ void k_pos_grad(const float* __restrict__ dX0, float* __restrict__ dPos, int B, int T) {
  int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= T * kD) return;
  int b0 = blockIdx.y * kPosRows, b1 = min(B, b0 + kPosRows);
  float s = 0.f;
  for (int b = b0; b < b1; ++b) s += dX0[(int64_t)b * T * kD + e];
  atomicAdd(dPos + e, s);
}
void launch_embed_bwd_reduce(const float* dX0, const float* dTgtHead, float* dTgtTotal, float* dPos, double* pos_normsq,
                             double* undedup, int B, int T, cudaStream_t st) { PAMREC_PROF("embed_bwd_reduce", 2, st);
  if (B == 0) return;
  k_dtgt_total<<<B, 128, 0, st>>>(dX0, dTgtHead, dTgtTotal, pos_normsq, undedup, T);
  dim3 grid((T * kD + 127) / 128, (B + kPosRows - 1) / kPosRows);
  k_pos_grad<<<grid, 128, 0, st>>>(dX0, dPos, B, T);
}

// ------------------------------------------------------------------------------------------
size_t sparse_temp_bytes(int64_t n_keys) {
  size_t a = 0, b = 0;
  int* p = nullptr;
  cub::DeviceRadixSort::SortPairs(nullptr, a, p, p, p, p, (int)n_keys, 0, 32, (cudaStream_t)0);
  cub::DeviceScan::InclusiveSum(nullptr, b, p, p, (int)n_keys, (cudaStream_t)0);
  return a > b ? a : b;
}

// world > 1: the key is the row's address in the sharded table, owner * rows_per_shard + local row (kernels_shard.cu)
__global__ void k_build_keys(const int* __restrict__ hist_ids, const int* __restrict__ tgt_ids, int64_t n_hist,
                             int64_t n_tgt, int world, int64_t rps, int* __restrict__ keys, int* __restrict__ idx) {
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_hist + n_tgt) return;
  int id = p < n_hist ? hist_ids[p] : tgt_ids[p - n_hist];
  keys[p] = world > 1 ? (int)((int64_t)(id % world) * rps + id / world) : id;
  idx[p] = (int)p;
}
__global__ void k_head_flags(const int* __restrict__ skeys, int64_t n, int* __restrict__ flags) {
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  flags[p] = (p == 0 || skeys[p] != skeys[p - 1]) ? 1 : 0;
}
__global__ void k_unique_fill(const int* __restrict__ skeys, const int* __restrict__ uidx, int64_t n,
                              int* __restrict__ ukeys, int* __restrict__ slot, int* __restrict__ nuniq) {
  int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  if (p == 0 || skeys[p] != skeys[p - 1]) {
    int u = uidx[p] - 1;
    ukeys[u] = skeys[p];
    if (slot != nullptr) slot[skeys[p]] = u;
  }
  if (p == n - 1) *nuniq = uidx[p];
}

__device__ __forceinline__ void atomic_add4(float* p, const float4& v) {
#if __CUDA_ARCH__ >= 900
  atomicAdd(reinterpret_cast<float4*>(p), v);
#else
  atomicAdd(p, v.x); atomicAdd(p + 1, v.y); atomicAdd(p + 2, v.z); atomicAdd(p + 3, v.w);
#endif
}

// Warp-level segmented reduction over sorted positions.  A warp walks `iters` consecutive blocks of 32 positions and carries
// the sum of the run that is still open at lane 31 into the next block, so a run of equal keys costs one red.global.add per
// warp walk instead of one per 32 positions: with a Zipf id distribution (and the padding id 0 in every short history) the
// hottest rows own runs of 10^5..10^6 positions and their atomics on a single 64-byte line were the whole kernel time.
template <int W>
__global__ void __launch_bounds__(256)
k_seg_reduce(const int* __restrict__ skeys, const int* __restrict__ sidx, const int* __restrict__ uidx, int64_t n,
             int64_t n_hist, const float* __restrict__ hist_grad, int hist_ld, int hist_col,
             const float* __restrict__ tgt_grad, int tgt_ld, int tgt_col, float* __restrict__ accum,
             double* __restrict__ normsq, int iters) {
  constexpr int CH = W / 4;
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32 * iters;
  float4 carry[CH];
#pragma unroll
  for (int c = 0; c < CH; ++c) carry[c] = f4_zero();
  int carry_key = 0, carry_u = 0;
  bool carry_open = false;                       // warp-uniform
  float sq = 0.f;
  for (int it = 0; it < iters; ++it) {
    const int64_t p = warp0 + (int64_t)it * 32 + lane;
    if (warp0 + (int64_t)it * 32 >= n) break;    // warp-uniform
    const bool valid = p < n;
    int key = INT_MAX - lane;                    // positions past the end: distinct keys above every real one
    const float* row = nullptr;
    int u = 0;
    if (valid) {
      key = skeys[p];
      const int src = sidx[p];
      row = src < n_hist ? hist_grad + (int64_t)src * hist_ld + hist_col
                         : tgt_grad + (int64_t)(src - n_hist) * tgt_ld + tgt_col;
      u = uidx[p] - 1;
    }
    const int key0 = __shfl_sync(0xffffffffu, key, 0);
    if (carry_open && key0 != carry_key) {       // the open run ended exactly at the block boundary
      if (lane == 0) {
#pragma unroll
        for (int c = 0; c < CH; ++c) atomic_add4(accum + (int64_t)carry_u * W + 4 * c, carry[c]);
      }
      carry_open = false;
    }
    const bool joins_carry = carry_open && key == carry_key;       // keys are sorted: lanes 0..k of the block
    const int key_next = __shfl_down_sync(0xffffffffu, key, 1);
    const bool tail = valid && lane < 31 && key_next != key;        // lane 31 stays open until the next block decides
    float4 gl[CH];                                                  // the whole row first: CH independent 16-byte loads in flight
#pragma unroll
    for (int c = 0; c < CH; ++c) gl[c] = valid ? ld4(row + 4 * c) : f4_zero();
#pragma unroll
    for (int c = 0; c < CH; ++c) {
      float4 g = gl[c];
      sq += f4_dot(g, g);
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        float4 o;
        o.x = __shfl_up_sync(0xffffffffu, g.x, d); o.y = __shfl_up_sync(0xffffffffu, g.y, d);
        o.z = __shfl_up_sync(0xffffffffu, g.z, d); o.w = __shfl_up_sync(0xffffffffu, g.w, d);
        const int ko = __shfl_up_sync(0xffffffffu, key, d);
        if (lane >= d && ko == key) { g.x += o.x; g.y += o.y; g.z += o.z; g.w += o.w; }
      }
      if (joins_carry) { g.x += carry[c].x; g.y += carry[c].y; g.z += carry[c].z; g.w += carry[c].w; }
      if (tail) atomic_add4(accum + (int64_t)u * W + 4 * c, g);
      carry[c].x = __shfl_sync(0xffffffffu, g.x, 31); carry[c].y = __shfl_sync(0xffffffffu, g.y, 31);
      carry[c].z = __shfl_sync(0xffffffffu, g.z, 31); carry[c].w = __shfl_sync(0xffffffffu, g.w, 31);
    }
    carry_key = __shfl_sync(0xffffffffu, key, 31);
    carry_u = __shfl_sync(0xffffffffu, u, 31);
    carry_open = __shfl_sync(0xffffffffu, valid ? 1 : 0, 31) != 0;
  }
  if (carry_open && lane == 0) {
#pragma unroll
    for (int c = 0; c < CH; ++c) atomic_add4(accum + (int64_t)carry_u * W + 4 * c, carry[c]);
  }
  const double s = warp_sum_d((double)sq);
  if (lane == 0 && s != 0.0) atomicAdd(normsq, s);
}

// keys (history ids then target ids) -> sorted -> unique list (ukeys, nuniq), rank of every position (uidx) and,
// when the table has a slot map, row -> unique index.  key_range = number of distinct key values.
int launch_sparse_plan(const SparseTable& t, const int* hist_ids, const int* tgt_ids, int64_t n_hist, int64_t n_tgt,
                       int world, int64_t rps, int64_t key_range, bool fill_slot, void* cub_temp, size_t cub_bytes,
                       cudaStream_t st) { PAMREC_PROF("sparse_plan", 3, st);
  const int64_t n = n_hist + n_tgt;
  if (n == 0) { cudaMemsetAsync(t.nuniq, 0, sizeof(int), st); return 0; }
  const unsigned g256 = (unsigned)((n + 255) / 256);
  k_build_keys<<<g256, 256, 0, st>>>(hist_ids, tgt_ids, n_hist, n_tgt, world, rps, t.keys, t.idx);
  int bits = 1;
  while (bits < 31 && ((int64_t)1 << bits) < key_range) ++bits;
  size_t bytes = cub_bytes;
  if (cub::DeviceRadixSort::SortPairs(cub_temp, bytes, t.keys, t.skeys, t.idx, t.sidx, (int)n, 0, bits, st) != cudaSuccess)
    return -1;
  k_head_flags<<<g256, 256, 0, st>>>(t.skeys, n, t.keys);          // keys buffer reused as head flags
  bytes = cub_bytes;
  if (cub::DeviceScan::InclusiveSum(cub_temp, bytes, t.keys, t.uidx, (int)n, st) != cudaSuccess) return -1;
  k_unique_fill<<<g256, 256, 0, st>>>(t.skeys, t.uidx, n, t.ukeys, fill_slot ? t.slot : nullptr, t.nuniq);
  return 0;
}

// duplicate rows summed into accum[unique index]; normsq += sum of squares of every (un-deduplicated) row
int launch_sparse_segreduce(const SparseTable& t, int64_t n, int64_t n_hist, const float* hist_grad, int hist_ld, int hist_col,
                            const float* tgt_grad, int tgt_ld, int tgt_col, double* normsq, cudaStream_t st) {
  PAMREC_PROF("sparse_segreduce", 1, st);
  if (t.width != 4 && t.width != 8 && t.width != 16 && t.width != 32) return -1;
  if (n == 0) return 0;
  cudaMemsetAsync(t.accum, 0, (size_t)n * t.width * sizeof(float), st);
  // blocks of 32 positions per warp walk: 1 while the grid would not fill the GPU otherwise, up to 16 for large batches
  int64_t iters = n / (148 * 8 * 8 * 32);
  iters = iters < 1 ? 1 : (iters > 16 ? 16 : iters);
  const int64_t per_cta = 8 * 32 * iters;                        // 8 warps per CTA
  const unsigned gw = (unsigned)((n + per_cta - 1) / per_cta);
#define PAMREC_SEG_REDUCE(W)                                                                                                   \
  k_seg_reduce<W><<<gw, 256, 0, st>>>(t.skeys, t.sidx, t.uidx, n, n_hist, hist_grad, hist_ld, hist_col, tgt_grad, tgt_ld, tgt_col, \
                                      t.accum, normsq, (int)iters)
  switch (t.width) {
    case 16: PAMREC_SEG_REDUCE(16); break;
    case 4: PAMREC_SEG_REDUCE(4); break;
    case 32: PAMREC_SEG_REDUCE(32); break;
    default: PAMREC_SEG_REDUCE(8); break;
  }
#undef PAMREC_SEG_REDUCE
  return 0;
}

// L2 rows of the unique ids (sequential_base_model.py:647-664, pamrec.py:173-182)
template <int W>
__global__ void __launch_bounds__(256)
k_sparse_l2norm(const int* __restrict__ ukeys, const int* __restrict__ nuniq, const float* __restrict__ w, float l2,
                double* __restrict__ normsq, double* __restrict__ reg_acc, const int* __restrict__ has0) {
  __shared__ double sh[8];
  constexpr int CH = W / 4;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)(*nuniq) * CH;
  double s = 0.0;
  if (i < total) {
    int u = (int)(i / CH), c = (int)(i % CH);
    const int key = ukeys[u];
    float4 v = ld4(w + (int64_t)key * W + 4 * c);
    if (!(has0 != nullptr && key == 0 && *has0 == 0)) s = (double)f4_dot(v, v);   // row 0 looked up without being an L2 row (SparseTable::l2_has0)
  }
  s = warp_sum_d(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int k = 0; k < 8; ++k) tot += sh[k];
    if (tot != 0.0) {
      atomicAdd(normsq, (double)l2 * (double)l2 * tot);
      atomicAdd(reg_acc, 0.5 * (double)l2 * tot);
    }
  }
}
int launch_sparse_l2norm(const SparseTable& t, int64_t n_keys, float l2, double* reg_acc, cudaStream_t st) { PAMREC_PROF("sparse_l2norm", 1, st);
  int64_t total = n_keys * (t.width / 4);
  unsigned g = (unsigned)((total + 255) / 256);
#define PAMREC_L2NORM(W) k_sparse_l2norm<W><<<g, 256, 0, st>>>(t.ukeys, t.nuniq, t.w, l2, t.normsq, reg_acc, t.l2_has0)
  switch (t.width) {
    case 4: case 8: case 16: case 20: case 32: case 40: break;
    default: return -1;
  }
  if (total == 0) return 0;
  switch (t.width) {
    case 16: PAMREC_L2NORM(16); break;
    case 4: PAMREC_L2NORM(4); break;
    case 20: PAMREC_L2NORM(20); break;
    case 32: PAMREC_L2NORM(32); break;
    case 8: PAMREC_L2NORM(8); break;
    default: PAMREC_L2NORM(40); break;
  }
#undef PAMREC_L2NORM
  return 0;
}

__device__ __forceinline__ void adam_row4(float4& w, float4& m, float4& v, const float4& g, float lr, float b1, float b2,
                                          float eps) {
  // TF _apply_sparse_shared: m = m*b1 + g*(1-b1); v = v*b2 + g*g*(1-b2); w -= lr*m/(sqrt(v)+eps)
  m.x = m.x * b1 + g.x * (1.f - b1); m.y = m.y * b1 + g.y * (1.f - b1);
  m.z = m.z * b1 + g.z * (1.f - b1); m.w = m.w * b1 + g.w * (1.f - b1);
  v.x = v.x * b2 + (g.x * g.x) * (1.f - b2); v.y = v.y * b2 + (g.y * g.y) * (1.f - b2);
  v.z = v.z * b2 + (g.z * g.z) * (1.f - b2); v.w = v.w * b2 + (g.w * g.w) * (1.f - b2);
  w.x -= lr * m.x / (sqrtf(v.x) + eps); w.y -= lr * m.y / (sqrtf(v.y) + eps);
  w.z -= lr * m.z / (sqrtf(v.z) + eps); w.w -= lr * m.w / (sqrtf(v.w) + eps);
}
__device__ __forceinline__ float clip_scale(const double* normsq, float clip, int is_clip) {
  if (!is_clip) return 1.0f;
  float norm = (float)sqrt(*normsq);
  return clip / fmaxf(norm, clip);            // tf.clip_by_norm: t * clip / max(norm, clip)
}

// full-table sweep: the HBM-bound kernel (6 x row bytes per row + 4 B slot)
template <int W>
__global__ void __launch_bounds__(256)
k_table_adam_dense(float* __restrict__ tw, float* __restrict__ tm, float* __restrict__ tv, const int* __restrict__ slot,
                   const float* __restrict__ accum, const double* __restrict__ normsq, int64_t n_rows, float l2, float lr,
                   float b1, float b2, float eps, float clip, int is_clip, const int* __restrict__ has0) {
  constexpr int CH = W / 4;
  const int64_t total = n_rows * CH;
  const float scale = clip_scale(normsq, clip, is_clip);
  const bool no_l2_row0 = has0 != nullptr && *has0 == 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / CH;
    const int c = (int)(i % CH);
    float4 w = ld4(tw + 4 * i), m = ld4(tm + 4 * i), v = ld4(tv + 4 * i);
    float4 g = f4_zero();
    const int u = __ldg(slot + r);
    if (u >= 0) {
      float4 a = accum ? ld4(accum + (int64_t)u * W + 4 * c) : f4_zero();
      const float l2r = (no_l2_row0 && r == 0) ? 0.f : l2;
      g.x = scale * (a.x + l2r * w.x); g.y = scale * (a.y + l2r * w.y);
      g.z = scale * (a.z + l2r * w.z); g.w = scale * (a.w + l2r * w.w);
    }
    adam_row4(w, m, v, g, lr, b1, b2, eps);
    st4(tw + 4 * i, w); st4(tm + 4 * i, m); st4(tv + 4 * i, v);
  }
}
template <int W>
__global__ void __launch_bounds__(256)
k_table_adam_lazy(float* __restrict__ tw, float* __restrict__ tm, float* __restrict__ tv, const int* __restrict__ ukeys,
                  const int* __restrict__ nuniq, const float* __restrict__ accum, const double* __restrict__ normsq, float l2,
                  float lr, float b1, float b2, float eps, float clip, int is_clip, const int* __restrict__ has0) {
  constexpr int CH = W / 4;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)(*nuniq) * CH) return;
  const int u = (int)(i / CH), c = (int)(i % CH);
  const int64_t o = (int64_t)ukeys[u] * W + 4 * c;
  const float scale = clip_scale(normsq, clip, is_clip);
  if (has0 != nullptr && ukeys[u] == 0 && *has0 == 0) l2 = 0.f;
  float4 w = ld4(tw + o), m = ld4(tm + o), v = ld4(tv + o);
  float4 a = accum ? ld4(accum + (int64_t)u * W + 4 * c) : f4_zero();
  float4 g;
  g.x = scale * (a.x + l2 * w.x); g.y = scale * (a.y + l2 * w.y);
  g.z = scale * (a.z + l2 * w.z); g.w = scale * (a.w + l2 * w.w);
  adam_row4(w, m, v, g, lr, b1, b2, eps);
  st4(tw + o, w); st4(tm + o, m); st4(tv + o, v);
}
__global__ void k_slot_reset(const int* __restrict__ ukeys, const int* __restrict__ nuniq, int* __restrict__ slot) {
  int64_t u = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u < *nuniq) slot[ukeys[u]] = -1;
}

template <int W>
static void sparse_adam_w(const SparseTable& t, int64_t n_keys, int mode, float l2, float lr, float b1, float b2, float eps,
                          float clip, int is_clip, cudaStream_t st) {
  if (mode == PAMREC_ADAM_DENSE_EXACT) {
    int64_t total = t.n_rows * (W / 4);
    int64_t blocks = (total + 255) / 256;
    const int64_t cap = 148 * 32;                                 // grid-stride above 32 CTAs per SM
    unsigned g = (unsigned)(blocks < cap ? blocks : cap);
    k_table_adam_dense<W><<<g, 256, 0, st>>>(t.w, t.m, t.v, t.slot, t.accum, t.normsq, t.n_rows, l2, lr, b1, b2, eps, clip, is_clip, t.l2_has0);
  } else {
    int64_t total = n_keys * (W / 4);
    if (total == 0) return;
    k_table_adam_lazy<W><<<(unsigned)((total + 255) / 256), 256, 0, st>>>(t.w, t.m, t.v, t.ukeys, t.nuniq, t.accum, t.normsq, l2,
                                                                        lr, b1, b2, eps, clip, is_clip, t.l2_has0);
  }
}
int launch_sparse_adam(const SparseTable& t, int64_t n_keys, int mode, float l2, float lr_t, float b1, float b2, float eps,
                       float clip, int is_clip, cudaStream_t st) { PAMREC_PROF("sparse_adam", 1, st);
  switch (t.width) {
    case 16: sparse_adam_w<16>(t, n_keys, mode, l2, lr_t, b1, b2, eps, clip, is_clip, st); break;
    case 4: sparse_adam_w<4>(t, n_keys, mode, l2, lr_t, b1, b2, eps, clip, is_clip, st); break;
    case 20: sparse_adam_w<20>(t, n_keys, mode, l2, lr_t, b1, b2, eps, clip, is_clip, st); break;
    case 32: sparse_adam_w<32>(t, n_keys, mode, l2, lr_t, b1, b2, eps, clip, is_clip, st); break;
    case 8: sparse_adam_w<8>(t, n_keys, mode, l2, lr_t, b1, b2, eps, clip, is_clip, st); break;
    case 40: sparse_adam_w<40>(t, n_keys, mode, l2, lr_t, b1, b2, eps, clip, is_clip, st); break;
    default: return -1;
  }
  return 0;
}
void launch_slot_reset(const SparseTable& t, int64_t n_keys, cudaStream_t st) { PAMREC_PROF("slot_reset", 1, st);
  if (n_keys == 0) return;
  k_slot_reset<<<(unsigned)((n_keys + 255) / 256), 256, 0, st>>>(t.ukeys, t.nuniq, t.slot);
}

// ------------------------------------------------------------------------------------------
// dense variables: |g + l2 p|^2 and the L2 loss term per TF variable; a variable is cut into kNormSplit pieces (the largest -
// the [10, 1600] time-aware tables - would otherwise keep one CTA busy for 60 dependent iterations), partial sums by atomics
constexpr int kNormSplit = 8;
__global__ void __launch_bounds__(256)
k_dense_norm(const float* __restrict__ P, const float* __restrict__ G, const int* __restrict__ seg_tab, float layer_l2,
             double* __restrict__ seg_normsq, const double* __restrict__ pos_normsq, double* __restrict__ reg_acc) {
  __shared__ double sh[2][8];
  const int s = blockIdx.x;
  const int64_t off = seg_tab[4 * s];
  const int n = seg_tab[4 * s + 1], flags = seg_tab[4 * s + 2];
  const float l2 = (flags & PAMREC_SEG_L2) ? layer_l2 : 0.f;
  const int per = ((n + kNormSplit - 1) / kNormSplit + 3) & ~3;
  const int i0 = blockIdx.y * per, i1 = min(n, i0 + per);
  if (i0 >= n && blockIdx.y > 0) return;
  double a = 0.0, b = 0.0;
#pragma unroll 4
  for (int i = i0 + threadIdx.x; i < i1; i += 256) {
    float p = P[off + i];
    float g = G[off + i] + l2 * p;
    a += (double)g * (double)g;
    b += (double)p * (double)p;
  }
  a = warp_sum_d(a); b = warp_sum_d(b);
  if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = a; sh[1][threadIdx.x >> 5] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ta = 0.0, tb = 0.0;
    for (int k = 0; k < 8; ++k) { ta += sh[0][k]; tb += sh[1][k]; }
    if (flags & PAMREC_SEG_POS) { if (blockIdx.y == 0) seg_normsq[s] = *pos_normsq; }      // sparse-style norm of the position table
    else if (ta != 0.0) atomicAdd(seg_normsq + s, ta);
    if (l2 != 0.f && tb != 0.0) atomicAdd(reg_acc, 0.5 * (double)l2 * tb);
  }
}
void launch_dense_norm(const float* P, const float* G, const int* seg_tab, int n_seg, float layer_l2, double* seg_normsq,
                       const double* pos_normsq, double* reg_acc, cudaStream_t st) { PAMREC_PROF("dense_norm", 1, st);
  cudaMemsetAsync(seg_normsq, 0, (size_t)n_seg * sizeof(double), st);
  k_dense_norm<<<dim3(n_seg, kNormSplit), 256, 0, st>>>(P, G, seg_tab, layer_l2, seg_normsq, pos_normsq, reg_acc);
}

__global__ void __launch_bounds__(256)
k_dense_adam(float* __restrict__ P, const float* __restrict__ G, float* __restrict__ M, float* __restrict__ V,
             const int* __restrict__ seg_id, const int* __restrict__ seg_tab, const double* __restrict__ seg_normsq, int64_t n,
             float layer_l2, float lr, const float* __restrict__ lr_dev, float b1, float b2, float eps, float clip, int is_clip) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (lr_dev != nullptr) lr = __ldg(lr_dev);
  const int s = seg_id[i];
  const int flags = seg_tab[4 * s + 2];
  const float l2 = (flags & PAMREC_SEG_L2) ? layer_l2 : 0.f;
  float p = P[i];
  float g = G[i] + l2 * p;
  if (is_clip) {
    float norm = (float)sqrt(seg_normsq[s]);
    g = g * clip / fmaxf(norm, clip);
  }
  float m = M[i], v = V[i];
  if (flags & PAMREC_SEG_POS) {           // IndexedSlices variable: sparse apply form
    m = m * b1 + g * (1.f - b1);
    v = v * b2 + (g * g) * (1.f - b2);
  } else {                                // ApplyAdam kernel form
    m += (g - m) * (1.f - b1);
    v += (g * g - v) * (1.f - b2);
  }
  p -= lr * m / (sqrtf(v) + eps);
  P[i] = p; M[i] = m; V[i] = v;
}
void launch_dense_adam(float* P, const float* G, float* M, float* V, const int* seg_id, const int* seg_tab,
                       const double* seg_normsq, int64_t n, float layer_l2, float lr_t, const float* lr_dev, float b1, float b2, float eps,
                       float clip, int is_clip, cudaStream_t st) { PAMREC_PROF("dense_adam", 1, st);
  k_dense_adam<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P, G, M, V, seg_id, seg_tab, seg_normsq, n, layer_l2, lr_t, lr_dev, b1, b2,
                                                           eps, clip, is_clip);
}

__global__ void k_adam_step(long long step, double* __restrict__ step_dev, float lr, float b1, float b2, float* __restrict__ lr_out) {
  const double t = step > 0 ? (double)step : *step_dev + 1.0;
  *step_dev = t;
  *lr_out = (float)((double)lr * sqrt(1.0 - pow((double)b2, t)) / (1.0 - pow((double)b1, t)));
}
void launch_adam_step(int64_t step, double* step_dev, float lr, float b1, float b2, float* lr_out, cudaStream_t st) {
  PAMREC_PROF("adam_step", 1, st);
  k_adam_step<<<1, 1, 0, st>>>((long long)step, step_dev, lr, b1, b2, lr_out);
}

__global__ void k_finish_losses(const double* __restrict__ acc, float* __restrict__ losses, const double* __restrict__ l2sq,
                                float embed_l2, double* __restrict__ sp_normsq) {
  // pamrec.py:444-448 order: loss, data_loss, regular_loss, auxiliary_data_loss, order_loss
  double reg = acc[3];
  if (l2sq != nullptr) {
    reg += 0.5 * (double)embed_l2 * (l2sq[0] + l2sq[1] + l2sq[2] + l2sq[3]);
    for (int t = 0; t < 4; ++t) sp_normsq[t] += (double)embed_l2 * (double)embed_l2 * l2sq[t];
  }
  losses[0] = (float)(acc[0] + reg + acc[1] + acc[2]);
  losses[1] = (float)acc[0];
  losses[2] = (float)reg;
  losses[3] = (float)acc[1];
  losses[4] = (float)acc[2];
}
void launch_finish_losses(const double* loss_acc, float* losses, const double* l2sq, float embed_l2, double* sp_normsq, cudaStream_t st) {
  PAMREC_PROF("finish_losses", 1, st);
  k_finish_losses<<<1, 1, 0, st>>>(loss_acc, losses, l2sq, embed_l2, sp_normsq);
}

}  // namespace pamrec
