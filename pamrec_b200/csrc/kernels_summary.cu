// Device histograms of fp32 tensors for TensorBoard summaries (tf.summary.histogram / tensorflow/core/lib/histogram/histogram.cc):
// the default bucket limits, the bucket rule upper_bound(limits, (double)x), min / max / num / sum / sum_squares in double, and
// EncodeToProto(preserve_zero_buckets = false)'s compaction, so that the host copies only the compacted runs.
//
// Three launches per call:
//   k_hist_bin       one CTA per work item (a segment's range of at most kHistChunk elements): shared-memory bucket counts,
//                    flushed with one global atomic per non-empty bucket; per-CTA partial sums / min / max / non-finite count
//   k_hist_finalize  one CTA per segment: reduces its partials in a fixed order (two runs give identical bytes)
//   k_hist_compact   one CTA per segment: the non-empty buckets and the last limit of every run of empty ones
// A caller that sums the counts and statistics over ranks does so between the second and the third launch.
#include "kernels.h"

namespace pamrec {

namespace {

constexpr int kThreads = 256;
constexpr int kPerThread = (kHistBuckets + kThreads - 1) / kThreads;   // buckets per thread in the compaction scan

// buckets counted per value: #{p <= x} of the positive limits p_k = 1e-12 * 1.1^k (x >= 0, so -0 and 0 land in the 1e-12
// bucket), or #{p < |x|} (x < 0).  The estimate from log2 is within one of the answer; the exact double limits settle it.
__device__ __forceinline__ int hist_bucket(float x, const double* __restrict__ pos) {
  const float ax = fabsf(x);
  int k = (int)((__log2f(ax) + 39.86313713864835f) * 7.272540897341713f) + 1;   // 1 + log_1.1(ax / 1e-12)
  k = min(max(k, 0), kHistPos);
  const double d = (double)ax;
  if (x >= 0.f) {
    while (k < kHistPos && pos[k] <= d) ++k;
    while (k > 0 && pos[k - 1] > d) --k;
    return kHistZero + 1 + k;
  }
  while (k < kHistPos && pos[k] < d) ++k;
  while (k > 0 && pos[k - 1] >= d) --k;
  return kHistZero - k;
}

struct Acc {
  double sum = 0.0, sq = 0.0;
  float mn = INFINITY, mx = -INFINITY;
  int bad = 0;
};

// every lane of the warp calls this (valid = false for lanes past the end): equal buckets of a warp share one shared atomic
__device__ __forceinline__ void hist_add(float x, bool valid, const double* pos, int* cnt, Acc& a) {
  int b = -1;
  if (valid) {
    if (isfinite(x)) {
      const double d = (double)x;
      a.sum += d;
      a.sq += d * d;
      a.mn = fminf(a.mn, x);
      a.mx = fmaxf(a.mx, x);
      b = hist_bucket(x, pos);
    } else {
      ++a.bad;
    }
  }
  const unsigned same = __match_any_sync(0xffffffffu, b);
  if (b >= 0 && (threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(&cnt[b], __popc(same));
}

__device__ __forceinline__ int segment_of(const HistArgs& a, int item) {
  int lo = 0, hi = a.n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) / 2;
    if (a.first_item[mid] <= item) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// fixed-order block reduction of (sum, sq, mn, mx, bad); the result is valid in thread 0
__device__ void block_reduce(Acc& a) {
  __shared__ double s_sum[kThreads / 32], s_sq[kThreads / 32];
  __shared__ float s_mn[kThreads / 32], s_mx[kThreads / 32];
  __shared__ int s_bad[kThreads / 32];
  for (int o = 16; o; o >>= 1) {
    a.sum += __shfl_down_sync(0xffffffffu, a.sum, o);
    a.sq += __shfl_down_sync(0xffffffffu, a.sq, o);
    a.mn = fminf(a.mn, __shfl_down_sync(0xffffffffu, a.mn, o));
    a.mx = fmaxf(a.mx, __shfl_down_sync(0xffffffffu, a.mx, o));
    a.bad += __shfl_down_sync(0xffffffffu, a.bad, o);
  }
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) { s_sum[w] = a.sum; s_sq[w] = a.sq; s_mn[w] = a.mn; s_mx[w] = a.mx; s_bad[w] = a.bad; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < kThreads / 32; ++i) {
      a.sum += s_sum[i]; a.sq += s_sq[i]; a.mn = fminf(a.mn, s_mn[i]); a.mx = fmaxf(a.mx, s_mx[i]); a.bad += s_bad[i];
    }
  }
}

__global__ void __launch_bounds__(kThreads) k_hist_bin(const __grid_constant__ HistArgs a, int* __restrict__ bins,
                                                       double* __restrict__ part) {
  __shared__ double pos[kHistPos];
  __shared__ int cnt[kHistBuckets];
  for (int i = threadIdx.x; i < kHistPos; i += kThreads) pos[i] = a.pos[i];
  for (int i = threadIdx.x; i < kHistBuckets; i += kThreads) cnt[i] = 0;
  __syncthreads();
  const int item = blockIdx.x;
  const int s = segment_of(a, item);
  const int64_t begin = (int64_t)(item - a.first_item[s]) * kHistChunk;
  const int64_t n = min((int64_t)kHistChunk, a.count[s] - begin);
  const float* p = a.ptr[s] + begin;
  Acc acc;
  int64_t done = 0;
  if ((reinterpret_cast<uintptr_t>(p) & 15) == 0) {
    // two float4 loads in flight per thread; the trip count is the same for every thread, so whole warps reach hist_add
    const int64_t nv = n / 4;
    const float4* p4 = reinterpret_cast<const float4*>(p);
    for (int64_t base = 0; base < nv; base += 2 * kThreads) {
      const int64_t i0 = base + threadIdx.x, i1 = i0 + kThreads;
      const bool v0 = i0 < nv, v1 = i1 < nv;
      const float4 q0 = v0 ? __ldcs(p4 + i0) : make_float4(0.f, 0.f, 0.f, 0.f);
      const float4 q1 = v1 ? __ldcs(p4 + i1) : make_float4(0.f, 0.f, 0.f, 0.f);
      hist_add(q0.x, v0, pos, cnt, acc); hist_add(q0.y, v0, pos, cnt, acc);
      hist_add(q0.z, v0, pos, cnt, acc); hist_add(q0.w, v0, pos, cnt, acc);
      hist_add(q1.x, v1, pos, cnt, acc); hist_add(q1.y, v1, pos, cnt, acc);
      hist_add(q1.z, v1, pos, cnt, acc); hist_add(q1.w, v1, pos, cnt, acc);
    }
    done = nv * 4;
  }
  for (int64_t base = done; base < n; base += kThreads) {
    const int64_t i = base + threadIdx.x;
    const bool v = i < n;
    hist_add(v ? p[i] : 0.f, v, pos, cnt, acc);
  }
  __syncthreads();
  int* out = bins + (int64_t)s * kHistBuckets;
  for (int i = threadIdx.x; i < kHistBuckets; i += kThreads)
    if (cnt[i]) atomicAdd(out + i, cnt[i]);
  block_reduce(acc);
  if (threadIdx.x == 0) {
    double* q = part + (int64_t)item * 5;
    q[0] = acc.sum; q[1] = acc.sq; q[2] = (double)acc.mn; q[3] = (double)acc.mx; q[4] = (double)acc.bad;
  }
}

__global__ void __launch_bounds__(kThreads) k_hist_finalize(const __grid_constant__ HistArgs a, const double* __restrict__ part,
                                                            double* __restrict__ stats) {
  const int s = blockIdx.x;
  Acc acc;
  for (int it = a.first_item[s] + threadIdx.x; it < a.first_item[s + 1]; it += kThreads) {
    const double* q = part + (int64_t)it * 5;
    acc.sum += q[0]; acc.sq += q[1]; acc.mn = fminf(acc.mn, (float)q[2]); acc.mx = fmaxf(acc.mx, (float)q[3]); acc.bad += (int)q[4];
  }
  block_reduce(acc);
  const int sw = hist_stats_width(a.world);
  double* st = stats + (int64_t)s * sw;
  for (int i = threadIdx.x; i < sw; i += kThreads) st[i] = 0.0;
  __syncthreads();
  if (threadIdx.x == 0) {
    const bool any = acc.mn <= acc.mx;                         // an empty histogram keeps TF's Clear() values
    st[HIST_NUM] = (double)(a.count[s] - acc.bad);
    st[HIST_SUM] = acc.sum;
    st[HIST_SUM_SQUARES] = acc.sq;
    st[HIST_NONFINITE] = (double)acc.bad;
    st[HIST_SLOTS + a.rank] = any ? (double)acc.mn : DBL_MAX;
    st[HIST_SLOTS + a.world + a.rank] = any ? (double)acc.mx : -DBL_MAX;
  }
}

__global__ void __launch_bounds__(kThreads) k_hist_compact(const __grid_constant__ HistArgs a, const int* __restrict__ bins,
                                                           double* __restrict__ stats, double* __restrict__ out) {
  __shared__ int cnt[kHistBuckets];
  __shared__ int warp_tot[kThreads / 32];
  const int s = blockIdx.x;
  const int* c = bins + (int64_t)s * kHistBuckets;
  for (int i = threadIdx.x; i < kHistBuckets; i += kThreads) cnt[i] = c[i];
  __syncthreads();
  const int b0 = threadIdx.x * kPerThread;
  int mine = 0;
  for (int b = b0; b < b0 + kPerThread && b < kHistBuckets; ++b) mine += hist_emits(cnt, b) ? 1 : 0;
  // exclusive block scan of `mine`
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int incl = mine;
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += y;
  }
  if (lane == 31) warp_tot[w] = incl;
  __syncthreads();
  int at = incl - mine;
  for (int i = 0; i < w; ++i) at += warp_tot[i];
  const int64_t off = a.out_off[s], cap = a.out_off[s + 1] - a.out_off[s];
  for (int b = b0; b < b0 + kPerThread && b < kHistBuckets; ++b) {
    if (!hist_emits(cnt, b)) continue;
    if (at < cap) {
      out[2 * (off + at)] = hist_limit(a.pos, b);
      out[2 * (off + at) + 1] = (double)cnt[b];
    }
    ++at;
  }
  if (threadIdx.x == kThreads - 1) stats[(int64_t)s * hist_stats_width(a.world) + HIST_LEN] = (double)at;
}

}  // namespace

const double* hist_positive_limits() {
  // InitDefaultBuckets: v = 1e-12, then v *= 1.1 in double while v < 1e20 (repeated products, bit-identical to TF's table)
  struct Table {
    double pos[kHistPos];
    bool ok;
    Table() {
      double v = 1.0e-12;
      int k = 0;
      while (v < 1.0e20 && k < kHistPos) { pos[k++] = v; v *= 1.1; }
      ok = k == kHistPos && !(v < 1.0e20);
    }
  };
  static const Table t;
  return t.ok ? t.pos : nullptr;
}

int64_t hist_items(int64_t count) { return (count + kHistChunk - 1) / kHistChunk; }

void launch_hist_bin(const HistArgs& a, int total_items, int* bins, double* part, double* stats, cudaStream_t st) {
  PAMREC_PROF("hist_bin", 2, st);
  if (total_items > 0) k_hist_bin<<<total_items, kThreads, 0, st>>>(a, bins, part);
  k_hist_finalize<<<a.n, kThreads, 0, st>>>(a, part, stats);
}

void launch_hist_compact(const HistArgs& a, const int* bins, double* stats, double* out, cudaStream_t st) {
  PAMREC_PROF("hist_compact", 1, st);
  k_hist_compact<<<a.n, kThreads, 0, st>>>(a, bins, stats, out);
}

}  // namespace pamrec
