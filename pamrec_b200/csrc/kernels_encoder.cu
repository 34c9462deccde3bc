// Encoder kernels: embedding gather, bucket planning, time-aware Q/K/V projection,
// key-masked attention, LayerNorm + point-wise FFN — forward and backward.
//
// Token-parallel kernels (projection, FFN): a CTA owns a tile of kTokTile = 64 token rows (40 floats each, shared-memory row
// stride 44), warp w the rows 16w .. 16w+15, and every [tokens x 40] x [40 x 40] contraction - forward, input gradient
// and weight gradient - runs on the tensor cores as an error-compensated 3xTF32 mma.sync (mma.cuh); LayerNorm and
// its backward are evaluated in the MMA fragment layout (row sums are 4-lane shuffles).  Tokens are bucket-sorted
// first so that a CTA needs exactly one (Wq,Wk,Wv)[bucket] triple: the reference instead materialises a
// [B,T,40,40] gather per matrix (pamrec.py:714-728).  Attention beyond T = 128 (up to there: kernels_attn_mma.cu): one thread
// per query row, see k_attn_fwd.
#include "kernels.h"
#include "mma.cuh"

namespace pamrec {

// ------------------------------------------------------------------------------------------
// G1+G2+G3+X1 (sequential_base_model.py:603-616,666-668; pamrec.py:155-159,251-257):
// x0[b,t,:] = item[ih[b,t]] | cate[ch[b,t]] | item[items[b]] | cate[cates[b]]  +  pos[t]
// One thread per 16-byte chunk, kEmbU tokens per thread.  A CTA of 320 threads covers 32 x kEmbU tokens: phase 1
// stages the four ids and the position of every token in shared memory (coalesced 4-byte loads), phase 2 issues all
// kEmbU row loads of a thread back to back (they are independent, so kEmbU x 16 B per thread are in flight while
// HBM answers: the kernel is bound by bytes in flight, not by instruction issue), phase 3 adds the L1-resident
// position row and writes; a warp's stores are contiguous 512 B.
constexpr int kEmbU = 8;
constexpr int kEmbTok = 32;
__global__ void __launch_bounds__(kEmbTok * 10, 3)
k_embed_fwd(const int* __restrict__ ih, const int* __restrict__ ch, const int* __restrict__ items,
            const int* __restrict__ cates, const float* __restrict__ item_w, const float* __restrict__ cate_w,
            const float* __restrict__ pos, float* __restrict__ x0, float* __restrict__ tgt, int64_t n_tok, int T) {
  constexpr int TOK = kEmbTok * kEmbU;
  __shared__ int s_id[4][TOK];      // history item, history cate, target item, target cate
  __shared__ int s_t[TOK];
  const int tid = threadIdx.x;
  const int64_t tok0 = (int64_t)blockIdx.x * TOK;
  for (int i = tid; i < TOK; i += kEmbTok * 10) {
    const int64_t tok = tok0 + i;
    if (tok < n_tok) {
      const int64_t b = tok / T;
      s_t[i] = (int)(tok - b * T);
      s_id[0][i] = __ldg(ih + tok);
      s_id[1][i] = __ldg(ch + tok);
      s_id[2][i] = __ldg(items + b);
      s_id[3][i] = __ldg(cates + b);
    }
  }
  __syncthreads();
  const int c = tid % 10, tl = tid / 10;
  const int which = c < 4 ? 0 : (c == 4 ? 1 : (c < 9 ? 2 : 3));
  const bool is_item = (which & 1) == 0;
  const int sub = c < 4 ? c : (c < 9 && c > 4 ? c - 5 : 0);
  const float* table = is_item ? item_w : cate_w;
  const int width = is_item ? kI : kC;
  float4 v[kEmbU];
#pragma unroll
  for (int j = 0; j < kEmbU; ++j) {
    const int i = j * kEmbTok + tl;
    if (tok0 + i < n_tok) v[j] = __ldg(reinterpret_cast<const float4*>(table + (int64_t)s_id[which][i] * width) + sub);
  }
#pragma unroll
  for (int j = 0; j < kEmbU; ++j) {
    const int i = j * kEmbTok + tl;
    const int64_t tok = tok0 + i;
    if (tok < n_tok) {
      const int t = s_t[i];
      if (tgt != nullptr && t == 0 && c >= 5) st4(tgt + (tok / T) * kE + 4 * (c - 5), v[j]);
      const float4 p = __ldg(reinterpret_cast<const float4*>(pos + t * kD) + c);
      float4 o = v[j];
      o.x += p.x; o.y += p.y; o.z += p.z; o.w += p.w;
      st4(x0 + tok * kD + 4 * c, o);
    }
  }
}

void launch_embed_fwd(const int* ih, const int* ch, const int* items, const int* cates, const float* item_w,
                      const float* cate_w, const float* pos, float* x0, float* tgt, int64_t n_rows, int T,
                      cudaStream_t st) {
  PAMREC_PROF("embed_fwd", 1, st);
  const int64_t n_tok = n_rows * T;
  if (n_tok == 0) return;
  const int64_t per_cta = (int64_t)kEmbU * kEmbTok;
  k_embed_fwd<<<(unsigned)((n_tok + per_cta - 1) / per_cta), kEmbTok * 10, 0, st>>>(ih, ch, items, cates, item_w, cate_w, pos, x0,
                                                                                  tgt, n_tok, T);
}

// ------------------------------------------------------------------------------------------
// Bucket planning: counting sort of tokens by play-ratio bucket and a tile table.  Bins 0..9 are the rows of the time-aware
// tables; bin kZeroBin holds every token whose bucket id lies outside 0..9 (lisan gives 10 for a ratio beyond its last border,
// or for a zero duration).  The reference gathers those tokens' matrices with tf.gather on the GPU, which returns a zero row
// for an out-of-range index: their Q, K and V are 0 and they add nothing to the tables' gradients (k_proj_fwd / k_proj_bwd).
// ctl: [0..15] counts, [16..31] cursors, [32] number of tiles.
constexpr int kZeroBin = kNB;
constexpr int kBins = kNB + 1;
__global__ void k_bucket_hist(const float* __restrict__ lt, int n, int* __restrict__ bucket, int* __restrict__ ctl) {
  __shared__ int h[16];
  if (threadIdx.x < 16) h[threadIdx.x] = 0;
  __syncthreads();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    // tf.cast(float -> int32) truncates (pamrec.py:716): ids 0..9 are the values in (-1, 10); NaN falls out of range too
    const float v = lt[i];
    const int k = (v > -1.f && v < (float)kNB) ? (int)v : kZeroBin;
    bucket[i] = k;
    atomicAdd(&h[k], 1);
  }
  __syncthreads();
  if (threadIdx.x < kBins && h[threadIdx.x]) atomicAdd(&ctl[threadIdx.x], h[threadIdx.x]);
}

__global__ void k_bucket_plan(int* __restrict__ ctl, int* __restrict__ tile_bucket, int* __restrict__ tile_begin,
                              int* __restrict__ tile_count) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  int start = 0, nt = 0;
  for (int k = 0; k < kBins; ++k) {
    int cnt = ctl[k];
    ctl[16 + k] = start;
    for (int o = 0; o < cnt; o += kTokTile) {
      tile_bucket[nt] = k;
      tile_begin[nt] = start + o;
      tile_count[nt] = min(kTokTile, cnt - o);
      ++nt;
    }
    start += cnt;
  }
  ctl[32] = nt;
}

__global__ void k_bucket_scatter(const int* __restrict__ bucket, int n, int* __restrict__ ctl, int* __restrict__ perm) {
  __shared__ int h[16], base[16];
  if (threadIdx.x < 16) h[threadIdx.x] = 0;
  __syncthreads();
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int k = -1, r = 0;
  if (i < n) { k = bucket[i]; r = atomicAdd(&h[k], 1); }
  __syncthreads();
  if (threadIdx.x < kBins) base[threadIdx.x] = h[threadIdx.x] ? atomicAdd(&ctl[16 + threadIdx.x], h[threadIdx.x]) : 0;
  __syncthreads();
  if (i < n) perm[base[k] + r] = i;
}

void launch_bucket_plan(const float* lt, int n, int* bucket, int* perm, int* ctl, int* tile_bucket, int* tile_begin,
                        int* tile_count, cudaStream_t st) {
  PAMREC_PROF("bucket_plan", 3, st);
  cudaMemsetAsync(ctl, 0, 64 * sizeof(int), st);
  if (n == 0) return;
  int g = (n + 255) / 256;
  k_bucket_hist<<<g, 256, 0, st>>>(lt, n, bucket, ctl);
  k_bucket_plan<<<1, 32, 0, st>>>(ctl, tile_bucket, tile_begin, tile_count);
  k_bucket_scatter<<<g, 256, 0, st>>>(bucket, n, ctl, perm);
}

// ------------------------------------------------------------------------------------------
constexpr int kTileIt = (kTokTile * 10 + kTokThreads - 1) / kTokThreads;   // float4 per thread for a full token tile

// ------------------------------------------------------------------------------------------
// N1 + A1 forward: qin = LN_a(x); Q = qin Wq[k], K = x Wk[k], V = x Wv[k]   (pamrec.py:521-522,714-728)
// One bucket-sorted tile of up to kTokTile tokens per CTA, three 3xTF32 tensor-core GEMMs per warp (kWarpRows tokens each).
// (definitions of kTS, load_split_mat, load_tile44, ln_row44 are further down with the FFN kernels)
constexpr int kTS = 44;
__device__ __forceinline__ void load_split_mat(uint32_t* __restrict__ hi, uint32_t* __restrict__ lo, const float* __restrict__ W, int tid);
__device__ __forceinline__ void load_tile44(float* __restrict__ dst, const float* __restrict__ src, const int* toks, int cnt, int tid);
constexpr int kLnWriteF = 1, kLnWriteXhat = 2;
__device__ __forceinline__ void ln_row44(float* __restrict__ row, const float* __restrict__ beta, const float* __restrict__ gamma,
                                         float& mean, float& rstd, int write);
__device__ __forceinline__ void store_frag_rows(float* __restrict__ dst, const float (&c)[kMT][5][4], int64_t tok0, const int* toks,
                                                int row_base, int cnt, int lane);

constexpr int kProjFwdSmem = (6 * kDD + 2 * kTokTile * kTS + 2 * kD) * 4;
__global__ void __launch_bounds__(kTokThreads)
k_proj_fwd(const float* __restrict__ X, const int* __restrict__ perm, const int* __restrict__ ctl,
           const int* __restrict__ tile_bucket, const int* __restrict__ tile_begin, const int* __restrict__ tile_count,
           const float* __restrict__ Wq, const float* __restrict__ Wk, const float* __restrict__ Wv,
           const float* __restrict__ ln_beta, const float* __restrict__ ln_gamma, float* __restrict__ QIN,
           float* __restrict__ Q, float* __restrict__ K, float* __restrict__ V) {
  int tile = blockIdx.x;
  if (tile >= ctl[32]) return;
  extern __shared__ __align__(16) float sm[];
  uint32_t* Whi = reinterpret_cast<uint32_t*>(sm);          // q | k | v
  uint32_t* Wlo = Whi + 3 * kDD;
  float* xs = sm + 6 * kDD;                                 // x
  float* qs = xs + kTokTile * kTS;                          // qin = LN_a(x)
  float* lnp = qs + kTokTile * kTS;                         // beta | gamma
  __shared__ int toks[kTokTile];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int k = tile_bucket[tile], begin = tile_begin[tile], cnt = tile_count[tile];
  const bool zero = k == kZeroBin;                          // zero matrices: Q = K = V = 0, qin as for any token
  load_split_mat(Whi, Wlo, zero ? nullptr : Wq + (int64_t)k * kDD, tid);
  load_split_mat(Whi + kDD, Wlo + kDD, zero ? nullptr : Wk + (int64_t)k * kDD, tid);
  load_split_mat(Whi + 2 * kDD, Wlo + 2 * kDD, zero ? nullptr : Wv + (int64_t)k * kDD, tid);
  if (tid < kD) { lnp[tid] = ln_beta[tid]; lnp[kD + tid] = ln_gamma[tid]; }
  if (tid < cnt) toks[tid] = perm[begin + tid];
  __syncthreads();
  load_tile44(xs, X, toks, cnt, tid);
  __syncthreads();
  if (tid < kTokTile) {
    // thread r: row r.  qin row -> shared (A operand of the Q GEMM) and -> global
    float* xr = xs + tid * kTS;
    float* qr = qs + tid * kTS;
#pragma unroll
    for (int i = 0; i < 10; ++i) st4(qr + 4 * i, ld4(xr + 4 * i));
    float mean, rstd;
    ln_row44(qr, lnp, lnp + kD, mean, rstd, kLnWriteF);
    if (tid < cnt) {
      float* o = QIN + (int64_t)toks[tid] * kD;
#pragma unroll
      for (int i = 0; i < 10; ++i) st4(o + 4 * i, ld4(qr + 4 * i));
    }
  }
  __syncthreads();
  const float* xw = xs + kWarpRows * w * kTS;
  const float* qw = qs + kWarpRows * w * kTS;
#pragma unroll 1
  for (int m = 0; m < 3; ++m) {
    float c[kMT][5][4];
#pragma unroll
    for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
      for (int nt = 0; nt < 5; ++nt)
#pragma unroll
        for (int q = 0; q < 4; ++q) c[mt][nt][q] = 0.f;
    const float* aw = m == 0 ? qw : xw;
    warp_gemm_rows_x40x40<kMT, false>(c, [&](int r, int kk) { return aw[r * kTS + kk]; }, Whi + m * kDD, Wlo + m * kDD, lane);
    store_frag_rows(m == 0 ? Q : (m == 1 ? K : V), c, 0, toks, kWarpRows * w, cnt, lane);
  }
}

void launch_proj_fwd(const float* X, const int* perm, const int* ctl, const int* tile_bucket, const int* tile_begin,
                     const int* tile_count, int max_tiles, const float* Wq, const float* Wk, const float* Wv,
                     const float* ln_beta, const float* ln_gamma, float* QIN, float* Q, float* K, float* V,
                     cudaStream_t st) {
  PAMREC_PROF("proj_fwd", 1, st);
  k_proj_fwd<<<max_tiles, kTokThreads, kProjFwdSmem, st>>>(X, perm, ctl, tile_bucket, tile_begin, tile_count, Wq, Wk, Wv,
                                                        ln_beta, ln_gamma, QIN, Q, K, V);
}

// ------------------------------------------------------------------------------------------
// A2-A4 forward: P = softmax_j(mask ? Q K^T / sqrt(40) : -(2^32)+1);  y = P V + qin  (pamrec.py:768-810)
//
// ONE THREAD == ONE QUERY ROW.  The 40 query values, the 40 output accumulators and a chunk of 8 scores live in
// registers; every lane of a warp reads the SAME key / value row from shared memory (a broadcast: one wavefront per
// LDS.128, no bank conflicts, no shuffles), so a key costs 20 LDS.128 for 80 FMAs and the 40 independent FMA chains
// hide the latency at low occupancy.  Scores go through a chunked online softmax (one rescale per 8 keys); the row
// maximum m and the row sum l are saved for the backward pass.  NW warps serve one sample, SPB samples share a CTA.
constexpr int kAttnCh = 8;
__host__ __device__ inline int attn_nw(int T) { return (T + 31) / 32; }
__host__ __device__ inline int attn_spb(int T) { int nw = attn_nw(T); return nw >= 4 ? 1 : 4 / nw; }
// floats per sample (16-byte multiple): K | V | mask [T4] | indices of the live keys [T4] | their count [4]
__host__ __device__ inline int attn_fwd_per(int T) { return 2 * T * kAttnStride + 2 * ((T + 3) & ~3) + 4; }
// The keys a query attends to are the sample's live ones: a masked key's weight is exp(-(2^32) - m) = 0 exactly whenever the sample
// has any live key, so both attention kernels walk a compacted index list (built once per sample by one warp) instead of testing
// the mask per key - half of the score / PV work at the bench's uniform history lengths.  lv / nl: list and count in shared memory.
__device__ __forceinline__ void attn_live_list(const int* __restrict__ mk, int T, int lane, int* __restrict__ lv, int* __restrict__ nl) {
  int base = 0;
  for (int c = 0; c < T; c += 32) {
    const int j = c + lane;
    const bool live = j < T && mk[j] != 0;
    const unsigned bal = __ballot_sync(0xffffffffu, live);
    if (live) lv[base + __popc(bal & ((1u << lane) - 1u))] = j;
    base += __popc(bal);
  }
  if (lane == 0) *nl = base;
}
inline size_t attn_fwd_smem(int T) { return (size_t)attn_spb(T) * attn_fwd_per(T) * 4; }

// 40-wide dot product as four independent FMA chains of ten (a single chain of 40 would serialise on FMA latency)
__device__ __forceinline__ float dot40(const float4 (&q)[10], const float* __restrict__ row) {
  float4 r = ld4(row);
  float4 a = make_float4(q[0].x * r.x, q[0].y * r.y, q[0].z * r.z, q[0].w * r.w);
#pragma unroll
  for (int i = 1; i < 10; ++i) {
    r = ld4(row + 4 * i);
    a.x = fmaf(q[i].x, r.x, a.x); a.y = fmaf(q[i].y, r.y, a.y); a.z = fmaf(q[i].z, r.z, a.z); a.w = fmaf(q[i].w, r.w, a.w);
  }
  return (a.x + a.y) + (a.z + a.w);
}

__global__ void __launch_bounds__(256)
k_attn_fwd(const float* __restrict__ Q, const float* __restrict__ K, const float* __restrict__ V,
           const float* __restrict__ QIN, const int* __restrict__ mask, float* __restrict__ Y, float* __restrict__ PV,
           float* __restrict__ ML, int B, int T) {
  extern __shared__ __align__(16) float sm[];
  const int nw = attn_nw(T), spb = attn_spb(T), tps = nw * 32;
  const int per = attn_fwd_per(T);                          // floats per sample: K | V | mask
  const int tid = threadIdx.x;
  const int b0 = blockIdx.x * spb;
  const int ns = min(spb, B - b0);
  for (int i = tid; i < ns * T * 10; i += blockDim.x) {
    const int sl = i / (T * 10), rc = i % (T * 10), r = rc / 10, c = rc % 10;
    const int64_t g = ((int64_t)(b0 + sl) * T + r) * kD + 4 * c;
    float* base = sm + sl * per;
    st4(base + r * kAttnStride + 4 * c, ld4(K + g));
    st4(base + T * kAttnStride + r * kAttnStride + 4 * c, ld4(V + g));
  }
  for (int i = tid; i < ns * T; i += blockDim.x) {
    const int sl = i / T, r = i % T;
    reinterpret_cast<int*>(sm + sl * per + 2 * T * kAttnStride)[r] = mask[(int64_t)(b0 + sl) * T + r];
  }
  __syncthreads();
  const int sl = tid / tps, t = tid % tps;
  const int T4 = (T + 3) & ~3;
  if (sl < ns && t < 32) {                                   // the first warp of every sample (tps is a multiple of 32)
    int* mki = reinterpret_cast<int*>(sm + sl * per + 2 * T * kAttnStride);
    attn_live_list(mki, T, t, mki + T4, mki + 2 * T4);
  }
  __syncthreads();
  if (sl >= ns || t >= T) return;
  const float* Ks = sm + sl * per;
  const float* Vs = Ks + T * kAttnStride;
  const int* lv = reinterpret_cast<const int*>(Vs + T * kAttnStride) + T4;
  const int nl = lv[T4];
  const int64_t row = ((int64_t)(b0 + sl) * T + t) * kD;
  float4 q[10], o[10];
#pragma unroll
  for (int i = 0; i < 10; ++i) { q[i] = ld4(Q + row + 4 * i); o[i] = f4_zero(); }
  const float rscale = 1.0f / sqrtf((float)kD);
  float m = -INFINITY, l = 0.f;
  for (int k0 = 0; k0 < nl; k0 += kAttnCh) {
    float sc[kAttnCh];
    float cm = -INFINITY;
#pragma unroll
    for (int jj = 0; jj < kAttnCh; ++jj) {
      const int k = k0 + jj;
      float val = -INFINITY;
      if (k < nl) val = dot40(q, Ks + lv[k] * kAttnStride) * rscale;
      sc[jj] = val;
      cm = fmaxf(cm, val);
    }
    const float mn = fmaxf(m, cm);
    const float corr = expf(m - mn);                       // first chunk: exp(-inf) = 0 on empty accumulators
    l *= corr;
#pragma unroll
    for (int i = 0; i < 10; ++i) { o[i].x *= corr; o[i].y *= corr; o[i].z *= corr; o[i].w *= corr; }
#pragma unroll
    for (int jj = 0; jj < kAttnCh; ++jj) {
      const int k = k0 + jj;
      if (k < nl) {
        const float pj = expf(sc[jj] - mn);
        l += pj;
        const float* vr = Vs + lv[k] * kAttnStride;
#pragma unroll
        for (int i = 0; i < 10; ++i) f4_fma(o[i], pj, ld4(vr + 4 * i));
      }
    }
    m = mn;
  }
  if (nl == 0) {                                           // no live key at all: every score is the padding constant, uniform weights
    m = kMaskNeg; l = (float)T;
    for (int j = 0; j < T; ++j) {
#pragma unroll
      for (int i = 0; i < 10; ++i) f4_fma(o[i], 1.0f, ld4(Vs + j * kAttnStride + 4 * i));
    }
  }
  const float inv = 1.0f / l;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const float4 r = ld4(QIN + row + 4 * i);
    st4(Y + row + 4 * i, make_float4(fmaf(o[i].x, inv, r.x), fmaf(o[i].y, inv, r.y), fmaf(o[i].z, inv, r.z), fmaf(o[i].w, inv, r.w)));
    st4(PV + row + 4 * i, make_float4(o[i].x * inv, o[i].y * inv, o[i].z * inv, o[i].w * inv));
  }
  ML[2 * ((int64_t)(b0 + sl) * T + t)] = m;
  ML[2 * ((int64_t)(b0 + sl) * T + t) + 1] = l;
}

void launch_attn_fwd(const float* Q, const float* K, const float* V, const float* QIN, const int* mask, float* Y, float* PV,
                     float* ML, int B, int T, cudaStream_t st) {
  PAMREC_PROF("attn_fwd", 1, st);
  if (B == 0) return;
  const size_t smem = attn_fwd_smem(T);
  const int spb = attn_spb(T), threads = spb * attn_nw(T) * 32;
  k_attn_fwd<<<(B + spb - 1) / spb, threads, smem, st>>>(Q, K, V, QIN, mask, Y, PV, ML, B, T);
}

// ------------------------------------------------------------------------------------------
// Tensor-core token tiles (mma.cuh).  A CTA owns kTokTile consecutive tokens, warp w the rows kWarpRows*w ..; activation
// tiles live in shared memory with row stride 44 (16-byte aligned rows; the m16n8k8 A-fragment pattern (row g, column t)
// maps to banks 12g + t: conflict free), 40x40 weights as TF32 hi / lo halves with their natural stride 40.
// split a 40x40 fp32 matrix into TF32 halves in shared memory
__device__ __forceinline__ void load_split_mat(uint32_t* __restrict__ hi, uint32_t* __restrict__ lo, const float* __restrict__ W,
                                               int tid) {
  constexpr int IT = (kDD / 4 + kTokThreads - 1) / kTokThreads;   // 4
  float4 v[IT];
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int i = tid + it * kTokThreads;
    if (i < kDD / 4) v[it] = W != nullptr ? ld4(W + 4 * i) : f4_zero();
  }
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int i = tid + it * kTokThreads;
    if (i < kDD / 4) {
      uint4 h, l;
      split_tf32(v[it].x, h.x, l.x); split_tf32(v[it].y, h.y, l.y); split_tf32(v[it].z, h.z, l.z); split_tf32(v[it].w, h.w, l.w);
      *reinterpret_cast<uint4*>(hi + 4 * i) = h;
      *reinterpret_cast<uint4*>(lo + 4 * i) = l;
    }
  }
}
// rows [0, cnt) of a [*, 40] global matrix into a stride-44 tile, rows >= cnt zero-filled; toks == nullptr: consecutive rows
__device__ __forceinline__ void load_tile44(float* __restrict__ dst, const float* __restrict__ src, const int* toks, int cnt, int tid) {
  float4 v[kTileIt];
#pragma unroll
  for (int it = 0; it < kTileIt; ++it) {
    const int i = tid + it * kTokThreads;
    const int r = i / 10, c = i % 10;
    v[it] = f4_zero();
    if (r < cnt) v[it] = toks ? ld4(src + (int64_t)toks[r] * kD + 4 * c) : ld4(src + 4 * (int64_t)i);
  }
#pragma unroll
  for (int it = 0; it < kTileIt; ++it) {
    const int i = tid + it * kTokThreads;
    st4(dst + (i / 10) * kTS + 4 * (i % 10), v[it]);
  }
}
// LayerNorm of one stride-44 row held by one lane (pamrec.py:659-662): returns mean / rstd and rewrites the row in place
// as f = gamma * xhat + beta (kLnWriteF) or as xhat (kLnWriteXhat)
__device__ __forceinline__ void ln_row44(float* __restrict__ row, const float* __restrict__ beta, const float* __restrict__ gamma,
                                         float& mean, float& rstd, int write) {
  float4 x[10];
  float sacc = 0.f;
#pragma unroll
  for (int i = 0; i < 10; ++i) { x[i] = ld4(row + 4 * i); sacc += (x[i].x + x[i].y) + (x[i].z + x[i].w); }
  mean = sacc * (1.0f / kD);
  float v = 0.f;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    float a = x[i].x - mean, b = x[i].y - mean, c = x[i].z - mean, d = x[i].w - mean;
    v = fmaf(a, a, v); v = fmaf(b, b, v); v = fmaf(c, c, v); v = fmaf(d, d, v);
  }
  rstd = 1.0f / sqrtf(v * (1.0f / kD) + kLnEps);
  if (write == kLnWriteXhat) {
#pragma unroll
    for (int i = 0; i < 10; ++i)
      st4(row + 4 * i, make_float4((x[i].x - mean) * rstd, (x[i].y - mean) * rstd, (x[i].z - mean) * rstd, (x[i].w - mean) * rstd));
  } else if (write == kLnWriteF) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      const float4 g = ld4(gamma + 4 * i), b = ld4(beta + 4 * i);
      st4(row + 4 * i, make_float4(fmaf(g.x, (x[i].x - mean) * rstd, b.x), fmaf(g.y, (x[i].y - mean) * rstd, b.y),
                                   fmaf(g.z, (x[i].z - mean) * rstd, b.z), fmaf(g.w, (x[i].w - mean) * rstd, b.w)));
    }
  }
}

// ------------------------------------------------------------------------------------------
// N1 + F1 forward: f = LN_b(y); out = relu(f W1 + b1) W2 + b2 + f     (pamrec.py:534-535,565-577)
constexpr int kFfnFwdSmem = (4 * kDD + 2 * kTokTile * kTS + 4 * kD) * 4;
__global__ void __launch_bounds__(kTokThreads)
k_ffn_fwd(const float* __restrict__ Y, const float* __restrict__ W1, const float* __restrict__ b1,
          const float* __restrict__ W2, const float* __restrict__ b2, const float* __restrict__ ln_beta,
          const float* __restrict__ ln_gamma, float* __restrict__ OUT, float* __restrict__ Hdbg, int n_tok) {
  extern __shared__ __align__(16) float sm[];
  uint32_t* W1hi = reinterpret_cast<uint32_t*>(sm);
  uint32_t* W1lo = W1hi + kDD;
  uint32_t* W2hi = W1lo + kDD;
  uint32_t* W2lo = W2hi + kDD;
  float* fs = sm + 4 * kDD;                     // y, then f = LN(y)
  float* hs = fs + kTokTile * kTS;              // relu(f W1 + b1)
  float* pr = hs + kTokTile * kTS;              // b1 | b2 | beta | gamma
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int64_t tok0 = (int64_t)blockIdx.x * kTokTile;
  const int cnt = (int)min((int64_t)kTokTile, (int64_t)n_tok - tok0);
  load_split_mat(W1hi, W1lo, W1, tid);
  load_split_mat(W2hi, W2lo, W2, tid);
  if (tid < kD) { pr[tid] = b1[tid]; pr[kD + tid] = b2[tid]; pr[2 * kD + tid] = ln_beta[tid]; pr[3 * kD + tid] = ln_gamma[tid]; }
  load_tile44(fs, Y + tok0 * kD, nullptr, cnt, tid);
  __syncthreads();
  if (tid < kTokTile) {
    float mean, rstd;
    ln_row44(fs + tid * kTS, pr + 2 * kD, pr + 3 * kD, mean, rstd, kLnWriteF);  // thread r normalises row r
  }
  __syncthreads();
  const int g = lane >> 2, t = lane & 3;
  const float* fw = fs + kWarpRows * w * kTS;
  float* hw = hs + kWarpRows * w * kTS;
  float c[kMT][5][4];
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const float b0 = pr[8 * nt + 2 * t], bb1 = pr[8 * nt + 2 * t + 1];
      c[mt][nt][0] = b0; c[mt][nt][1] = bb1; c[mt][nt][2] = b0; c[mt][nt][3] = bb1;
    }
  warp_gemm_rows_x40x40<kMT, false>(c, [&](int r, int k) { return fw[r * kTS + k]; }, W1hi, W1lo, lane);
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const int r = 16 * mt + g, col = 8 * nt + 2 * t;
      *reinterpret_cast<float2*>(hw + r * kTS + col) = make_float2(fmaxf(c[mt][nt][0], 0.f), fmaxf(c[mt][nt][1], 0.f));
      *reinterpret_cast<float2*>(hw + (r + 8) * kTS + col) = make_float2(fmaxf(c[mt][nt][2], 0.f), fmaxf(c[mt][nt][3], 0.f));
    }
  __syncwarp();
  if (Hdbg != nullptr) {                        // test hook (PAMREC_DEBUG_SAVE_FFN_HIDDEN): the hidden activations as computed here
    for (int i = lane; i < kWarpRows * kD; i += 32) {
      const int r = i / kD, col = i % kD;
      if (kWarpRows * w + r < cnt) Hdbg[(tok0 + kWarpRows * w + r) * kD + col] = hw[r * kTS + col];
    }
  }
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const int r = 16 * mt + g, col = 8 * nt + 2 * t;
      const float2 f0 = *reinterpret_cast<const float2*>(fw + r * kTS + col);
      const float2 f1 = *reinterpret_cast<const float2*>(fw + (r + 8) * kTS + col);
      const float b0 = pr[kD + col], bb1 = pr[kD + col + 1];
      c[mt][nt][0] = b0 + f0.x; c[mt][nt][1] = bb1 + f0.y; c[mt][nt][2] = b0 + f1.x; c[mt][nt][3] = bb1 + f1.y;
    }
  warp_gemm_rows_x40x40<kMT, false>(c, [&](int r, int k) { return hw[r * kTS + k]; }, W2hi, W2lo, lane);
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const int r = kWarpRows * w + 16 * mt + g, col = 8 * nt + 2 * t;
      if (r < cnt) *reinterpret_cast<float2*>(OUT + (tok0 + r) * kD + col) = make_float2(c[mt][nt][0], c[mt][nt][1]);
      if (r + 8 < cnt) *reinterpret_cast<float2*>(OUT + (tok0 + r + 8) * kD + col) = make_float2(c[mt][nt][2], c[mt][nt][3]);
    }
}

void launch_ffn_fwd(const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                    const float* ln_beta, const float* ln_gamma, float* OUT, float* Hdbg, int n_tok, cudaStream_t st) {
  PAMREC_PROF("ffn_fwd", 1, st);
  if (n_tok == 0) return;
  k_ffn_fwd<<<(n_tok + kTokTile - 1) / kTokTile, kTokThreads, kFfnFwdSmem, st>>>(Y, W1, b1, W2, b2, ln_beta, ln_gamma, OUT, Hdbg, n_tok);
}

// ------------------------------------------------------------------------------------------
// shared pieces of the two backward kernels
// LayerNorm backward in C-fragment layout.  d[mt][nt][4] holds dF (grad wrt f = gamma * xhat + beta) of the warp's rows;
// xhat2(r, col) returns xhat[r][col .. col+1] of the warp's rows, rstd_w is their 1/std.  On return d holds dY (grad wrt the LN input); the column sums
// dbeta = sum dF and dgamma = sum dF * xhat of the warp's rows are added to red[0..39] / red[40..79] (shared memory).
template <typename XF>
__device__ __forceinline__ void ln_bwd_frag(float (&d)[kMT][5][4], XF xhat2, const float* __restrict__ rstd_w,
                                            const float* __restrict__ gamma, float* __restrict__ red, int lane) {
  const int g = lane >> 2, t = lane & 3;
  float sb[5][2], sg[5][2];
#pragma unroll
  for (int nt = 0; nt < 5; ++nt) { sb[nt][0] = sb[nt][1] = sg[nt][0] = sg[nt][1] = 0.f; }
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {                       // h = 0: row g, h = 1: row g + 8
      const int r = 16 * mt + g + 8 * h;
      float m1 = 0.f, m2 = 0.f;
      float xh[5][2];
#pragma unroll
      for (int nt = 0; nt < 5; ++nt) {
        const int col = 8 * nt + 2 * t;
        const float2 x = xhat2(r, col);                 // xhat[r][col], xhat[r][col + 1]
        xh[nt][0] = x.x; xh[nt][1] = x.y;
        const float d0 = d[mt][nt][2 * h], d1 = d[mt][nt][2 * h + 1];
        sb[nt][0] += d0; sb[nt][1] += d1;
        sg[nt][0] = fmaf(d0, x.x, sg[nt][0]); sg[nt][1] = fmaf(d1, x.y, sg[nt][1]);
        const float e0 = d0 * gamma[col], e1 = d1 * gamma[col + 1];
        m1 += e0 + e1;
        m2 = fmaf(e0, x.x, m2); m2 = fmaf(e1, x.y, m2);
      }
      m1 += __shfl_xor_sync(0xffffffffu, m1, 1); m1 += __shfl_xor_sync(0xffffffffu, m1, 2);
      m2 += __shfl_xor_sync(0xffffffffu, m2, 1); m2 += __shfl_xor_sync(0xffffffffu, m2, 2);
      m1 *= (1.0f / kD); m2 *= (1.0f / kD);
      const float rs = rstd_w[r];
#pragma unroll
      for (int nt = 0; nt < 5; ++nt) {
        const int col = 8 * nt + 2 * t;
        d[mt][nt][2 * h] = rs * (d[mt][nt][2 * h] * gamma[col] - m1 - xh[nt][0] * m2);
        d[mt][nt][2 * h + 1] = rs * (d[mt][nt][2 * h + 1] * gamma[col + 1] - m1 - xh[nt][1] * m2);
      }
    }
  }
#pragma unroll
  for (int nt = 0; nt < 5; ++nt)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      float a = sb[nt][j], b = sg[nt][j];
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
      if (g == 0) { atomicAdd(red + 8 * nt + 2 * t + j, a); atomicAdd(red + kD + 8 * nt + 2 * t + j, b); }
    }
}
// store the warp's 32 x 40 C fragments to rows tok0 + r (r < cnt) of a [*, 40] global matrix; toks != nullptr: permuted rows
__device__ __forceinline__ void store_frag_rows(float* __restrict__ dst, const float (&c)[kMT][5][4], int64_t tok0, const int* toks,
                                                int row_base, int cnt, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = row_base + 16 * mt + g + 8 * h;
      if (r < cnt) {
        float* o = dst + (toks ? (int64_t)toks[r] : tok0 + r) * kD + 2 * t;
#pragma unroll
        for (int nt = 0; nt < 5; ++nt) *reinterpret_cast<float2*>(o + 8 * nt) = make_float2(c[mt][nt][2 * h], c[mt][nt][2 * h + 1]);
      }
    }
}

// ------------------------------------------------------------------------------------------
// FFN + LN_b backward, input-gradient chain.  In: dOUT (grad of block output), Y.  Out: dY, the column sums dbeta / dgamma
// (one global atomic per element and CTA), and for the weight gradients (k_enc_dw, off the critical path) H = relu(f W1 + b1),
// DHR = dH o relu' and, when DOUT_KEEP is given, a copy of dOUT that outlives the buffer it came in.  Three 3xTF32 tensor-core
// GEMMs per token tile:   h = relu(f W1 + b1) [recomputed: its sign is relu'],  dH = dOUT W2^T,  dF = dOUT + (dH o relu') W1^T.
constexpr int kFfnBwdSmem = (4 * kDD + 3 * kTokTile * kTS + 4 * kD + 2 * kD + kTokTile) * 4;
__global__ void __launch_bounds__(kTokThreads)
k_ffn_bwd(const float* __restrict__ Y, const float* __restrict__ dOUT, const float* __restrict__ W1,
          const float* __restrict__ b1, const float* __restrict__ W2, const float* __restrict__ ln_beta,
          const float* __restrict__ ln_gamma, float* __restrict__ dY, float* __restrict__ H, float* __restrict__ DHR,
          float* __restrict__ DOUT_KEEP, float* __restrict__ dbeta, float* __restrict__ dgamma, int n_tok) {
  extern __shared__ __align__(16) float sm[];
  uint32_t* W1hi = reinterpret_cast<uint32_t*>(sm);
  uint32_t* W1lo = W1hi + kDD;
  uint32_t* W2hi = W1lo + kDD;
  uint32_t* W2lo = W2hi + kDD;
  float* xs = sm + 4 * kDD;                    // y, then xhat
  float* hs = xs + kTokTile * kTS;             // h = relu(f W1 + b1), later dH o relu'
  float* gs = hs + kTokTile * kTS;             // dOUT
  float* pr = gs + kTokTile * kTS;             // b1 | - | beta | gamma
  float* red = pr + 4 * kD;                    // dbeta | dgamma
  float* rstd_s = red + 2 * kD;                // per-row 1/std
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int64_t tok0 = (int64_t)blockIdx.x * kTokTile;
  const int cnt = (int)min((int64_t)kTokTile, (int64_t)n_tok - tok0);
  load_split_mat(W1hi, W1lo, W1, tid);
  load_split_mat(W2hi, W2lo, W2, tid);
  if (tid < kD) { pr[tid] = b1[tid]; pr[2 * kD + tid] = ln_beta[tid]; pr[3 * kD + tid] = ln_gamma[tid]; }
  if (tid < 2 * kD) red[tid] = 0.f;
  load_tile44(xs, Y + tok0 * kD, nullptr, cnt, tid);
  load_tile44(gs, dOUT + tok0 * kD, nullptr, cnt, tid);
  __syncthreads();
  if (tid < kTokTile) {
    float mean, rstd;
    ln_row44(xs + tid * kTS, pr + 2 * kD, pr + 3 * kD, mean, rstd, kLnWriteXhat);
    rstd_s[tid] = rstd;
  }
  if (DOUT_KEEP != nullptr)
    for (int i = tid; i < cnt * 10; i += kTokThreads) st4(DOUT_KEEP + (tok0 + i / 10) * kD + 4 * (i % 10), ld4(gs + (i / 10) * kTS + 4 * (i % 10)));
  __syncthreads();
  const float* xw = xs + kWarpRows * w * kTS;
  float* hw = hs + kWarpRows * w * kTS;
  const float* gw = gs + kWarpRows * w * kTS;
  const float* beta = pr + 2 * kD;
  const float* gamma = pr + 3 * kD;
  auto f_elem = [&](int r, int k) { return fmaf(gamma[k], xw[r * kTS + k], beta[k]); };
  float c[kMT][5][4];
  // ---- h = relu(f W1 + b1)
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const float b0 = pr[8 * nt + 2 * t], bb1 = pr[8 * nt + 2 * t + 1];
      c[mt][nt][0] = b0; c[mt][nt][1] = bb1; c[mt][nt][2] = b0; c[mt][nt][3] = bb1;
    }
  warp_gemm_rows_x40x40<kMT, false>(c, f_elem, W1hi, W1lo, lane);
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const int r = 16 * mt + g, col = 8 * nt + 2 * t;
#pragma unroll
      for (int q = 0; q < 4; ++q) c[mt][nt][q] = fmaxf(c[mt][nt][q], 0.f);
      *reinterpret_cast<float2*>(hw + r * kTS + col) = make_float2(c[mt][nt][0], c[mt][nt][1]);
      *reinterpret_cast<float2*>(hw + (r + 8) * kTS + col) = make_float2(c[mt][nt][2], c[mt][nt][3]);
    }
  store_frag_rows(H, c, tok0, nullptr, kWarpRows * w, cnt, lane);
  __syncwarp();
  // ---- dH = dOUT W2^T, masked by relu'
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt)
#pragma unroll
      for (int q = 0; q < 4; ++q) c[mt][nt][q] = 0.f;
  warp_gemm_rows_x40x40<kMT, true>(c, [&](int r, int k) { return gw[r * kTS + k]; }, W2hi, W2lo, lane);
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const int r = 16 * mt + g, col = 8 * nt + 2 * t;
      const float2 h0 = *reinterpret_cast<const float2*>(hw + r * kTS + col);
      const float2 h1 = *reinterpret_cast<const float2*>(hw + (r + 8) * kTS + col);
      if (!(h0.x > 0.f)) c[mt][nt][0] = 0.f;
      if (!(h0.y > 0.f)) c[mt][nt][1] = 0.f;
      if (!(h1.x > 0.f)) c[mt][nt][2] = 0.f;
      if (!(h1.y > 0.f)) c[mt][nt][3] = 0.f;
    }
  store_frag_rows(DHR, c, tok0, nullptr, kWarpRows * w, cnt, lane);
  __syncwarp();
  // ---- hs <- dH o relu'
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const int r = 16 * mt + g, col = 8 * nt + 2 * t;
      *reinterpret_cast<float2*>(hw + r * kTS + col) = make_float2(c[mt][nt][0], c[mt][nt][1]);
      *reinterpret_cast<float2*>(hw + (r + 8) * kTS + col) = make_float2(c[mt][nt][2], c[mt][nt][3]);
    }
  __syncwarp();
  // ---- dF = dOUT + (dH o relu') W1^T
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const int r = 16 * mt + g, col = 8 * nt + 2 * t;
      const float2 g0 = *reinterpret_cast<const float2*>(gw + r * kTS + col);
      const float2 g1 = *reinterpret_cast<const float2*>(gw + (r + 8) * kTS + col);
      c[mt][nt][0] = g0.x; c[mt][nt][1] = g0.y; c[mt][nt][2] = g1.x; c[mt][nt][3] = g1.y;
    }
  warp_gemm_rows_x40x40<kMT, true>(c, [&](int r, int k) { return hw[r * kTS + k]; }, W1hi, W1lo, lane);
  // ---- LN_b backward, dY out
  ln_bwd_frag(c, [&](int r, int col) { return *reinterpret_cast<const float2*>(xw + r * kTS + col); }, rstd_s + kWarpRows * w, gamma, red, lane);
  store_frag_rows(dY, c, tok0, nullptr, kWarpRows * w, cnt, lane);
  __syncthreads();
  if (tid < kD) { atomicAdd(dbeta + tid, red[tid]); atomicAdd(dgamma + tid, red[kD + tid]); }
}

void launch_ffn_bwd(const float* Y, const float* dOUT, const float* W1, const float* b1, const float* W2,
                    const float* ln_beta, const float* ln_gamma, float* dY, float* H, float* DHR, float* dOUT_keep,
                    float* dbeta, float* dgamma, int n_tok, cudaStream_t st) {
  PAMREC_PROF("ffn_bwd", 1, st);
  if (n_tok == 0) return;
  k_ffn_bwd<<<(n_tok + kTokTile - 1) / kTokTile, kTokThreads, kFfnBwdSmem, st>>>(Y, dOUT, W1, b1, W2, ln_beta, ln_gamma, dY, H, DHR,
                                                                             dOUT_keep, dbeta, dgamma, n_tok);
}

// ------------------------------------------------------------------------------------------
// Attention backward.  In: Q, K, V, dY (grad of y = P V + qin), the forward's y, qin and row statistics (m, l).
// Out: dQ, dK, dV.  Same thread mapping as the forward: with D_t = dy_t . (P V)_t (= sum_j p_tj dP_tj) known
// up front, pass A (thread == query row t) forms dQ_t in one sweep over the keys and pass B (thread == key j) forms
// dK_j and dV_j in one sweep over the queries; both recompute p = exp(s - m_t) / l_t from the saved statistics, all
// shared-memory reads are warp-wide broadcasts.
__host__ __device__ inline int attn_bwd_per(int T) { return 4 * T * kAttnStride + ((5 * T + 4 + 3) & ~3); }   // K | V | Q | dY | m | 1/l | D | mask | live list | count
inline size_t attn_bwd_smem(int T) { return (size_t)attn_spb(T) * attn_bwd_per(T) * 4; }

__global__ void __launch_bounds__(256)
k_attn_bwd(const float* __restrict__ Q, const float* __restrict__ K, const float* __restrict__ V,
           const float* __restrict__ dY, const float* __restrict__ PV,
           const float* __restrict__ ML, const int* __restrict__ mask, float* __restrict__ dQ, float* __restrict__ dK,
           float* __restrict__ dV, int B, int T) {
  extern __shared__ __align__(16) float sm[];
  const int nw = attn_nw(T), spb = attn_spb(T), tps = nw * 32;
  const int TS = T * kAttnStride;
  const int per = attn_bwd_per(T);
  const int tid = threadIdx.x;
  const int b0 = blockIdx.x * spb;
  const int ns = min(spb, B - b0);
  for (int i = tid; i < ns * T * 10; i += blockDim.x) {
    const int sl = i / (T * 10), rc = i % (T * 10), r = rc / 10, c = rc % 10;
    const int64_t g = ((int64_t)(b0 + sl) * T + r) * kD + 4 * c;
    float* base = sm + sl * per + r * kAttnStride + 4 * c;
    st4(base, ld4(K + g));
    st4(base + TS, ld4(V + g));
    st4(base + 2 * TS, ld4(Q + g));
    st4(base + 3 * TS, ld4(dY + g));
  }
  const int sl = tid / tps, t = tid % tps;
  const bool active = sl < ns && t < T;
  float* S = sm + sl * per;
  if (active) {
    const int64_t tok = (int64_t)(b0 + sl) * T + t;
    float d = 0.f;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      const float4 g = ld4(dY + tok * kD + 4 * i), o = ld4(PV + tok * kD + 4 * i);
      d = fmaf(g.x, o.x, d); d = fmaf(g.y, o.y, d); d = fmaf(g.z, o.z, d); d = fmaf(g.w, o.w, d);
    }
    S[4 * TS + t] = ML[2 * tok];
    S[4 * TS + T + t] = 1.0f / ML[2 * tok + 1];
    S[4 * TS + 2 * T + t] = d;
    reinterpret_cast<int*>(S + 4 * TS + 3 * T)[t] = mask[tok];
  }
  __syncthreads();
  if (sl < ns && t < 32) {
    int* mki = reinterpret_cast<int*>(S + 4 * TS + 3 * T);
    attn_live_list(mki, T, t, mki + T, mki + 2 * T);
  }
  __syncthreads();
  if (!active) return;
  const float* Ks = S;
  const float* Vs = S + TS;
  const float* Qs = S + 2 * TS;
  const float* Gs = S + 3 * TS;
  const float* rm = S + 4 * TS;
  const float* ril = rm + T;                               // 1 / row sum
  const float* rD = ril + T;
  const int* mk = reinterpret_cast<const int*>(rD + T);
  const int* lv = mk + T;
  const int nl = lv[T];
  const float rscale = 1.0f / sqrtf((float)kD);
  const int64_t row = ((int64_t)(b0 + sl) * T + t) * kD;
  // ---- pass A: dQ_t
  {
    float4 q[10], g[10], acc[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) { q[i] = ld4(Qs + t * kAttnStride + 4 * i); g[i] = ld4(Gs + t * kAttnStride + 4 * i); acc[i] = f4_zero(); }
    const float mt = rm[t], il = ril[t], Dt = rD[t];
#pragma unroll 2
    for (int k = 0; k < nl; ++k) {                         // live keys only: a masked key's score is a constant (dS = 0)
      const int j = lv[k];
      const float* kr = Ks + j * kAttnStride;
      const float sv = dot40(q, kr) * rscale;
      const float p = expf(sv - mt) * il;
      const float dp = dot40(g, Vs + j * kAttnStride);
      const float ds = p * (dp - Dt) * rscale;
#pragma unroll
      for (int i = 0; i < 10; ++i) f4_fma(acc[i], ds, ld4(kr + 4 * i));
    }
#pragma unroll
    for (int i = 0; i < 10; ++i) st4(dQ + row + 4 * i, acc[i]);
  }
  // ---- pass B: dK_j, dV_j  (this thread's row index now plays the key)
  {
    const int j = t;
    float4 kj[10], vj[10], ak[10], av[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) { kj[i] = ld4(Ks + j * kAttnStride + 4 * i); vj[i] = ld4(Vs + j * kAttnStride + 4 * i); ak[i] = f4_zero(); av[i] = f4_zero(); }
    const int mkj = mk[j];
    // a masked key of a sample that has live keys: p = exp(-(2^32) - m_t) = 0 for every query, nothing to accumulate (a warp whose
    // keys are all padding leaves here)
    const int tq_end = (mkj || nl == 0) ? T : 0;
    for (int tt = 0; tt < tq_end; ++tt) {
      const float* qr = Qs + tt * kAttnStride;
      const float* gr = Gs + tt * kAttnStride;
      const float sv = mkj ? dot40(kj, qr) * rscale : kMaskNeg;
      const float p = expf(sv - rm[tt]) * ril[tt];
      const float dp = dot40(vj, gr);
      const float ds = mkj ? p * (dp - rD[tt]) * rscale : 0.f;
#pragma unroll
      for (int i = 0; i < 10; ++i) { f4_fma(ak[i], ds, ld4(qr + 4 * i)); f4_fma(av[i], p, ld4(gr + 4 * i)); }
    }
#pragma unroll
    for (int i = 0; i < 10; ++i) { st4(dK + row + 4 * i, ak[i]); st4(dV + row + 4 * i, av[i]); }
  }
}

void launch_attn_bwd(const float* Q, const float* K, const float* V, const float* dY, const float* PV, const float* ML, const int* mask, float* dQ, float* dK, float* dV, int B, int T, cudaStream_t st) {
  PAMREC_PROF("attn_bwd", 1, st);
  if (B == 0) return;
  const size_t smem = attn_bwd_smem(T);
  const int spb = attn_spb(T), threads = spb * attn_nw(T) * 32;
  k_attn_bwd<<<(B + spb - 1) / spb, threads, smem, st>>>(Q, K, V, dY, PV, ML, mask, dQ, dK, dV, B, T);
}

// ------------------------------------------------------------------------------------------
// Projection + LN_a backward (bucket-sorted tiles), input-gradient chain.  In: X (block input), dY (residual path into qin),
// dQ, dK, dV.  Out: dX and the column sums dbeta, dgamma.  Three 3xTF32 tensor-core GEMMs per tile:
//   dqin = dY + dQ Wq^T,   dX = dK Wk^T + dV Wv^T + LN_a'(dqin).
// The table gradients dWq/dWk/dWv[bucket] are k_enc_dw's.
constexpr int kProjBwdSmem = (6 * kDD + 2 * kTokTile * kTS + 2 * kD + 2 * kD + 2 * kTokTile) * 4;
__global__ void __launch_bounds__(kTokThreads)
k_proj_bwd(const float* __restrict__ X, const float* __restrict__ dY, const float* __restrict__ dQ,
           const float* __restrict__ dK, const float* __restrict__ dV, const int* __restrict__ perm,
           const int* __restrict__ ctl, const int* __restrict__ tile_bucket, const int* __restrict__ tile_begin,
           const int* __restrict__ tile_count, const float* __restrict__ Wq, const float* __restrict__ Wk,
           const float* __restrict__ Wv, const float* __restrict__ ln_beta, const float* __restrict__ ln_gamma,
           float* __restrict__ dX, float* __restrict__ dbeta, float* __restrict__ dgamma) {
  int tile = blockIdx.x;
  if (tile >= ctl[32]) return;
  extern __shared__ __align__(16) float sm[];
  uint32_t* Whi = reinterpret_cast<uint32_t*>(sm);          // q | k | v
  uint32_t* Wlo = Whi + 3 * kDD;
  float* xs = sm + 6 * kDD;                                 // x (raw)
  float* gs = xs + kTokTile * kTS;                          // dQ, then dK, then dV
  float* lnp = gs + kTokTile * kTS;                         // beta | gamma
  float* red = lnp + 2 * kD;                                // dbeta | dgamma
  float* mean_s = red + 2 * kD;
  float* rstd_s = mean_s + kTokTile;
  __shared__ int toks[kTokTile];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int k = tile_bucket[tile], begin = tile_begin[tile], cnt = tile_count[tile];
  // zero matrices (bucket id outside 0..9): dX = LN_a'(dY) only
  const bool zero = k == kZeroBin;
  load_split_mat(Whi, Wlo, zero ? nullptr : Wq + (int64_t)k * kDD, tid);
  load_split_mat(Whi + kDD, Wlo + kDD, zero ? nullptr : Wk + (int64_t)k * kDD, tid);
  load_split_mat(Whi + 2 * kDD, Wlo + 2 * kDD, zero ? nullptr : Wv + (int64_t)k * kDD, tid);
  if (tid < kD) { lnp[tid] = ln_beta[tid]; lnp[kD + tid] = ln_gamma[tid]; }
  if (tid < 2 * kD) red[tid] = 0.f;
  if (tid < cnt) toks[tid] = perm[begin + tid];
  __syncthreads();
  load_tile44(xs, X, toks, cnt, tid);
  load_tile44(gs, dQ, toks, cnt, tid);
  __syncthreads();
  if (tid < kTokTile) {
    float mean, rstd;
    ln_row44(xs + tid * kTS, lnp, lnp + kD, mean, rstd, 0);
    mean_s[tid] = mean; rstd_s[tid] = rstd;
  }
  __syncthreads();
  const float* xw = xs + kWarpRows * w * kTS;
  const float* gw = gs + kWarpRows * w * kTS;
  const float* mw = mean_s + kWarpRows * w;
  const float* rw = rstd_s + kWarpRows * w;
  const float* gamma = lnp + kD;
  auto xhat = [&](int r, int i) { return (xw[r * kTS + i] - mw[r]) * rw[r]; };
  auto g_elem = [&](int r, int kk) { return gw[r * kTS + kk]; };
  float dqin[kMT][5][4], dx[kMT][5][4];
  // ---- dqin = dY + dQ Wq^T
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = kWarpRows * w + 16 * mt + g + 8 * h;
      const float* src = dY + (int64_t)toks[r < cnt ? r : 0] * kD + 2 * t;
#pragma unroll
      for (int nt = 0; nt < 5; ++nt) {
        const float2 v = r < cnt ? *reinterpret_cast<const float2*>(src + 8 * nt) : make_float2(0.f, 0.f);
        dqin[mt][nt][2 * h] = v.x; dqin[mt][nt][2 * h + 1] = v.y;
      }
    }
  warp_gemm_rows_x40x40<kMT, true>(dqin, g_elem, Whi, Wlo, lane);
  // ---- dX = dK Wk^T + dV Wv^T (+ LN backward below)
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt)
#pragma unroll
      for (int q = 0; q < 4; ++q) dx[mt][nt][q] = 0.f;
#pragma unroll 1
  for (int m = 1; m < 3; ++m) {
    __syncthreads();                                    // every warp is done with the previous gradient tile
    load_tile44(gs, m == 1 ? dK : dV, toks, cnt, tid);
    __syncthreads();
    warp_gemm_rows_x40x40<kMT, true>(dx, g_elem, Whi + m * kDD, Wlo + m * kDD, lane);
  }
  // ---- LN_a backward of dqin, added to dX
  ln_bwd_frag(dqin, [&](int r, int col) { return make_float2(xhat(r, col), xhat(r, col + 1)); }, rw, gamma, red, lane);
#pragma unroll
  for (int mt = 0; mt < kMT; ++mt)
#pragma unroll
    for (int nt = 0; nt < 5; ++nt)
#pragma unroll
      for (int q = 0; q < 4; ++q) dx[mt][nt][q] += dqin[mt][nt][q];
  store_frag_rows(dX, dx, 0, toks, kWarpRows * w, cnt, lane);
  __syncthreads();
  if (tid < kD) { atomicAdd(dbeta + tid, red[tid]); atomicAdd(dgamma + tid, red[kD + tid]); }
}

void launch_proj_bwd(const float* X, const float* dY, const float* dQ, const float* dK, const float* dV, const int* perm,
                     const int* ctl, const int* tile_bucket, const int* tile_begin, const int* tile_count, int max_tiles,
                     const float* Wq, const float* Wk, const float* Wv, const float* ln_beta, const float* ln_gamma,
                     float* dX, float* dbeta, float* dgamma, cudaStream_t st) {
  PAMREC_PROF("proj_bwd", 1, st);
  k_proj_bwd<<<max_tiles, kTokThreads, kProjBwdSmem, st>>>(X, dY, dQ, dK, dV, perm, ctl, tile_bucket, tile_begin, tile_count, Wq,
                                                        Wk, Wv, ln_beta, ln_gamma, dX, dbeta, dgamma);
}

// ------------------------------------------------------------------------------------------
// Weight gradients of one encoder block.  Nothing reads them before the optimiser, so api.cu runs this kernel on the side
// stream, beside the rest of the encoder's backward pass, in two launches per block as soon as their inputs exist:
//   a.ffn:   [dW1; db1] = [f 1]^T (dH o relu'),  [dW2; db2] = [h 1]^T dOUT      over every token (f = LN_b(y) recomputed);
//   !a.ffn:  dWq[k] = qin^T dQ,  dWk[k] = x^T dK,  dWv[k] = x^T dV      over the tokens of bucket k (the zero bin adds nothing).
// The products of a launch (two FFN ones, or bucket x {q, k, v}) are laid end to end as one list of token rows, and CTA i takes
// the i-th of gridDim.x equal ranges of that list: one or a few long runs per CTA whatever the bucket sizes.  Over a run every warp keeps
// one 3xTF32 accumulator in registers (warp w: rows 16w .. 16w+15 of each 64-row tile; tiles double-buffered with cp.async);
// at the end of the run the warps' sums meet in shared memory and leave as one global atomic per element.
constexpr int kDwRun = 256;                                 // least tokens per CTA the grid is sized for
constexpr int kEncDwSmem = (4 * kTokTile * kTS + 41 * kD + 2 * kD) * 4;
__device__ __forceinline__ void cp_async16(float* dst, const float* src, bool valid) {   // !valid: 16 zero bytes
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(d), "l"(src), "r"(valid ? 16 : 0));
}
__global__ void __launch_bounds__(kTokThreads)
k_enc_dw(const EncDwArgs a) {
  extern __shared__ __align__(16) float sm[];               // [2 buffers][A | B][kTokTile][kTS] | acc [41][40] | beta | gamma
  float* acc = sm + 4 * kTokTile * kTS;
  float* lnp = acc + 41 * kD;
  __shared__ int s_cnt[kNB];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid < kD) { lnp[tid] = a.ln_beta[tid]; lnp[kD + tid] = a.ln_gamma[tid]; }
  if (tid < kNB) s_cnt[tid] = a.ctl[tid];
  __syncthreads();
  // products s in [s_lo, s_hi): 0, 1 the FFN ones, 2 + 3k + p bucket k of Q (p = 0), K (1), V (2)
  const int s_lo = a.ffn ? 0 : 2, s_hi = a.ffn ? 2 : 2 + 3 * kNB;
  int64_t total = 0;
  if (a.ffn) total = 2 * (int64_t)a.n_tok;
  else for (int k = 0; k < kNB; ++k) total += 3 * (int64_t)s_cnt[k];
  const int64_t chunk = (total + gridDim.x - 1) / gridDim.x;
  const int64_t lo = blockIdx.x * chunk, hi = min(total, lo + chunk);
  const int lr = tid >> 1, c0 = 5 * (tid & 1);              // this thread copies row lr, float4 chunks c0 .. c0+4, of A and B
  int64_t v = 0;
  int bin0 = 0;                                             // first perm index of bucket k
  for (int s = s_lo; s < s_hi && v < hi; ++s) {
    const int k = s < 2 ? -1 : (s - 2) / 3, p = s < 2 ? -1 : (s - 2) % 3;
    const int64_t len = s < 2 ? a.n_tok : s_cnt[k];
    const int64_t b = max(lo, v) - v, e = min(hi, v + len) - v;
    v += len;
    if (b < e) {
      const bool bias = s < 2;
      const float* A = s == 0 ? a.y : s == 1 ? a.h : p == 0 ? a.qin : a.x;
      const float* Bm = s == 0 ? a.dhr : s == 1 ? a.dout : p == 0 ? a.dQ : p == 1 ? a.dK : a.dV;
      const int* rows = bias ? nullptr : a.perm + bin0;
      float* dW = s == 0 ? a.dW1 : s == 1 ? a.dW2 : (p == 0 ? a.dWq : p == 1 ? a.dWk : a.dWv) + (int64_t)k * kDD;
      float* db = s == 0 ? a.db1 : a.db2;
      for (int i = tid; i < 41 * kD; i += kTokThreads) acc[i] = 0.f;
      float cw[3][5][4];
#pragma unroll
      for (int mt = 0; mt < 3; ++mt)
#pragma unroll
        for (int nt = 0; nt < 5; ++nt)
#pragma unroll
          for (int q = 0; q < 4; ++q) cw[mt][nt][q] = 0.f;
      auto row_of = [&](int64_t i) -> int64_t { return i < e ? (rows ? (int64_t)rows[i] : i) : -1; };
      auto issue = [&](int buf, int64_t r) {                // one cp.async group per tile; rows past the run are zero-filled
        float* da = sm + 2 * buf * kTokTile * kTS + lr * kTS + 4 * c0;
        const int64_t o = (r >= 0 ? r : 0) * kD + 4 * c0;
#pragma unroll
        for (int j = 0; j < 5; ++j) {
          cp_async16(da + 4 * j, A + o + 4 * j, r >= 0);
          cp_async16(da + kTokTile * kTS + 4 * j, Bm + o + 4 * j, r >= 0);
        }
        asm volatile("cp.async.commit_group;\n" ::);
      };
      issue(0, row_of(b + lr));
      int64_t nxt = row_of(b + kTokTile + lr);
      int buf = 0;
      for (int64_t t0 = b; t0 < e; t0 += kTokTile, buf ^= 1) {
        if (t0 + kTokTile < e) issue(buf ^ 1, nxt);
        else asm volatile("cp.async.commit_group;\n" ::);
        nxt = row_of(t0 + 2 * kTokTile + lr);
        asm volatile("cp.async.wait_group 1;\n" ::);
        __syncthreads();
        float* As = sm + 2 * buf * kTokTile * kTS;
        if (s == 0) {                                       // f = LN_b(y), row tid
          if (tid < kTokTile) { float mean, rstd; ln_row44(As + tid * kTS, lnp, lnp + kD, mean, rstd, kLnWriteF); }
          __syncthreads();
        }
        const float* aw = As + kWarpRows * w * kTS;
        const float* bw = aw + kTokTile * kTS;
        warp_gemm_tn_48x40(cw, kWarpRows, [&](int r, int i) { return i < kD ? aw[r * kTS + i] : (i == kD && bias ? 1.f : 0.f); },
                           [&](int r, int n) { return bw[r * kTS + n]; }, lane);
        __syncthreads();                                    // the buffer is refilled two tiles on
      }
      tn_flush_smem(cw, acc, lane, bias ? kD : kD - 1);
      __syncthreads();
      for (int i = tid; i < kDD; i += kTokThreads) atomicAdd(dW + i, acc[i]);
      if (bias && tid < kD) atomicAdd(db + tid, acc[kDD + tid]);
      __syncthreads();                                      // acc is cleared by the next run
    }
    if (p == 2) bin0 += s_cnt[k];
  }
}

void launch_enc_dw(const EncDwArgs& a, cudaStream_t st) {
  PAMREC_PROF("enc_dw", 1, st);
  if (a.n_tok == 0) return;
  int dev = 0, n_sm = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
  // about one wave at two CTAs per SM, and runs of at least kDwRun tokens when every token is in a table bucket
  const int64_t runs = ((a.ffn ? 2 : 3) * (int64_t)a.n_tok + kDwRun - 1) / kDwRun;
  const int grid = (int)(runs < 2 * n_sm ? runs : 2 * n_sm);
  k_enc_dw<<<grid, kTokThreads, kEncDwSmem, st>>>(a);
}

// Dynamic shared memory above 48 KB is an opt-in per kernel AND per device: pamrec_bind calls this on the handle's device, so
// that no launcher keeps process-wide "already done" state (a second device in the same process gets its own opt-in).
int init_encoder_kernels(int max_T) {
  cudaError_t e = cudaSuccess;
  auto set = [&](const void* fn, size_t bytes) {
    if (e == cudaSuccess) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  };
  set((const void*)k_proj_fwd, kProjFwdSmem);
  set((const void*)k_ffn_fwd, kFfnFwdSmem);
  set((const void*)k_ffn_bwd, kFfnBwdSmem);
  set((const void*)k_proj_bwd, kProjBwdSmem);
  set((const void*)k_enc_dw, kEncDwSmem);
  size_t af = 0, ab = 0;
  for (int T = 1; T <= max_T; ++T) { af = af > attn_fwd_smem(T) ? af : attn_fwd_smem(T); ab = ab > attn_bwd_smem(T) ? ab : attn_bwd_smem(T); }
  set((const void*)k_attn_fwd, af);
  set((const void*)k_attn_bwd, ab);
  return e == cudaSuccess ? 0 : -1;
}

}  // namespace pamrec
