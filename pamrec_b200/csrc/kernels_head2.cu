// The head (attention pooling, MMoE, towers, losses) ROW-STATIONARY: one persistent cooperative kernel per direction in which
// every CTA owns a contiguous range of samples and carries them through all layers; a third, ordinary kernel computes the weight
// gradients beside the encoder's backward pass.
//
// Why: every layer of the head is followed by a batch norm over the whole batch (pamrec.py:366-372, base_model.py:680-686), so a
// step has 6 + 6 points where every row must have been seen; in between the work is a few MFLOP.  The tile programs that ran
// here before (round 2, first half; profiles/r02_bench_coop4.json) re-distributed 32 x 32 output tiles over the grid in every phase: 31 M warp instructions for
// 3 M warp-FMAs of arithmetic, 8 + 10 barriers, 0.57 ms.  Here
//   * a CTA stages the (batch-normalised, rectified) inputs of its <= 8 rows in shared memory, a thread owns one OUTPUT COLUMN
//     and keeps the 8 row accumulators in registers: per k one coalesced weight load and two broadcast LDS.128 feed 8 FFMAs,
//     fp32 throughout, contraction in index order (results agree with the fp64 oracle to ~1e-7);
//   * the thread that owns a column owns its batch-norm sums as well: one fp64 atomic per column and CTA, no reduction tree;
//   * row-local steps (pooling, MMoE mixing, tower inputs, their backward) never leave the CTA, so barriers remain only at the
//     batch-norm points: 6 forward, 7 backward (the 7th separates the loss from the towers);
//   * the backward dX chain reads TRANSPOSED weights (written once per step into the workspace by the first backward phase),
//     so it is the same column kernel; dW = act(x)^T dz has no consumer before the optimiser and runs as k_head2_dw on the
//     side stream while the encoder's backward pass runs on the main stream.
// Grid barrier with a leader section (batch-norm finalize, moving statistics, gamma / beta gradients, data parallel: all-reduce
// of the fp64 sums through the NVLink peer mailboxes, leader_p2p) as before.
#include <cstdio>

#include "head2.h"

namespace pamrec {

namespace {

constexpr int kT2 = kHead2Threads;          // 512 threads, one CTA per SM
constexpr int kRC = 8;                       // rows per chunk (= accumulators per thread)
constexpr int kXS = 640;                     // staged input columns per chunk (largest: 500 expert + 128 gate pre-activations)
constexpr int kWBuf = 32768;                 // floats of next-phase weights held in shared memory (largest set: 32 640)
constexpr int kSlots = 25;                   // tokens in flight per pass of the score-MLP phases: 25 x 20 columns = 500 threads

// ---- memory-ordering helpers.  Spin loads are RELAXED: an acquire load makes the SM invalidate its whole L1 (CCTL.IVALL) after
// every poll, which starved the warps that were still working; the acquire happens once, by a fence, after the awaited value
// has been seen.
__device__ __forceinline__ void st_release_u32(unsigned* p, unsigned v) { asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void st_flag_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_flag_sys_relaxed(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_acq_rel_sys() { asm volatile("fence.acq_rel.sys;" ::: "memory"); }

// ---- batch norm on load
struct BnC { float mean, inv, ga, be; };
__device__ __forceinline__ BnC bn_c(const BnSet& s, int c) { return BnC{s.stat[2 * c], s.stat[2 * c + 1], s.gamma[c], s.beta[c]}; }
__device__ __forceinline__ float bn_act(float z, const BnC& k) { return fmaxf(fmaf(k.ga, (z - k.mean) * k.inv, k.be), 0.f); }
// backward: dz from dA (gradient wrt the rectified output) with the column's global sums S1 = sum dy, S2 = sum dy * xhat
struct BnB { float mean, inv, ga, be, s1n, s2n; };
__device__ __forceinline__ BnB bn_b(const BnSet& s, int c, double count) {
  return BnB{s.stat[2 * c], s.stat[2 * c + 1], s.gamma[c], s.beta[c], (float)(s.bsums[2 * c] / count), (float)(s.bsums[2 * c + 1] / count)};
}
__device__ __forceinline__ float bn_dz(float da, float z, const BnB& k) {
  const float xh = (z - k.mean) * k.inv;
  const float dy = fmaf(k.ga, xh, k.be) > 0.f ? da : 0.f;
  return k.ga * k.inv * (dy - k.s1n - xh * k.s2n);
}

// ---- the column kernel: acc[r] += sum_k xs[(x_off + k) * 8 + r] * W[k * ldw]   (W already offset to the thread's column)
// (plain loads: the backward kernel reads transposed weights that its own first phase wrote)
__device__ __forceinline__ void col_gemm(const float* xs, int x_off, int K, const float* W, int ldw, float (&acc)[kRC]) {
  const float* x = xs + x_off * kRC;
#pragma unroll 8
  for (int k = 0; k < K; ++k) {
    const float w = W[(int64_t)k * ldw];
    const float4 a = ld4(x + k * kRC), b = ld4(x + k * kRC + 4);
    acc[0] = fmaf(a.x, w, acc[0]); acc[1] = fmaf(a.y, w, acc[1]); acc[2] = fmaf(a.z, w, acc[2]); acc[3] = fmaf(a.w, w, acc[3]);
    acc[4] = fmaf(b.x, w, acc[4]); acc[5] = fmaf(b.y, w, acc[5]); acc[6] = fmaf(b.z, w, acc[6]); acc[7] = fmaf(b.w, w, acc[7]);
  }
}
__device__ __forceinline__ void acc_set(float (&acc)[kRC], float v) {
#pragma unroll
  for (int r = 0; r < kRC; ++r) acc[r] = v;
}

// stage columns [0, C) of rows [row0, row0 + nr) of a row-major matrix into xs[(x_off + c) * 8 + r] through f(value, c); rows >= nr read as 0
template <typename F>
__device__ __forceinline__ void stage_cols(float* __restrict__ xs, int x_off, const float* __restrict__ src, int ld, int C, int64_t row0, int nr, F f) {
  for (int c = threadIdx.x; c < C; c += kT2) {
    float v[kRC];
#pragma unroll
    for (int r = 0; r < kRC; ++r) v[r] = r < nr ? src[(row0 + r) * ld + c] : 0.f;
    float o[kRC];
    f(c, v, o);
#pragma unroll
    for (int r = 0; r < kRC; ++r) if (r >= nr) o[r] = 0.f;
    st4(xs + (x_off + c) * kRC, make_float4(o[0], o[1], o[2], o[3]));
    st4(xs + (x_off + c) * kRC + 4, make_float4(o[4], o[5], o[6], o[7]));
  }
}
// forward staging: act = relu(bn(z)) of a pre-activation matrix
__device__ __forceinline__ void stage_act(float* xs, int x_off, const float* Z, int ld, int C, int64_t row0, int nr, const BnSet& s) {
  stage_cols(xs, x_off, Z, ld, C, row0, nr, [&](int c, const float (&v)[kRC], float (&o)[kRC]) {
    const BnC k = bn_c(s, c);
#pragma unroll
    for (int r = 0; r < kRC; ++r) o[r] = bn_act(v[r], k);
  });
}
// backward staging: dz = bn_bwd(dA, z); the buffer that held dA is overwritten with dz (k_head2_dw reads it)
__device__ __forceinline__ void stage_dz(float* xs, int x_off, float* dA, const float* Z, int ld, int C, int64_t row0, int nr, const BnSet& s, double count) {
  for (int c = threadIdx.x; c < C; c += kT2) {
    const BnB k = bn_b(s, c, count);
    float o[kRC];
#pragma unroll
    for (int r = 0; r < kRC; ++r) {
      o[r] = 0.f;
      if (r < nr) {
        const int64_t i = (row0 + r) * ld + c;
        o[r] = bn_dz(dA[i], Z[i], k);
        dA[i] = o[r];
      }
    }
    st4(xs + (x_off + c) * kRC, make_float4(o[0], o[1], o[2], o[3]));
    st4(xs + (x_off + c) * kRC + 4, make_float4(o[4], o[5], o[6], o[7]));
  }
}

// forward epilogue of a column: store z, add the rows to the column's batch-norm sums
__device__ __forceinline__ void epi_fwd(const float (&acc)[kRC], float* __restrict__ Z, int ld, int col, int64_t row0, int nr, double& s, double& q) {
#pragma unroll
  for (int r = 0; r < kRC; ++r)
    if (r < nr) { Z[(row0 + r) * ld + col] = acc[r]; s += (double)acc[r]; q += (double)acc[r] * (double)acc[r]; }
}
// backward epilogue: store dA (gradient wrt the rectified output of the layer whose pre-activations are Zp), add to its S1 / S2
__device__ __forceinline__ void epi_bwd(const float (&acc)[kRC], float* __restrict__ dA, const float* __restrict__ Zp, int ld, int col, int64_t row0, int nr,
                                        const BnC& k, double& s1, double& s2) {
#pragma unroll
  for (int r = 0; r < kRC; ++r)
    if (r < nr) {
      const int64_t i = (row0 + r) * ld + col;
      dA[i] = acc[r];
      const float xh = (Zp[i] - k.mean) * k.inv;
      const float dy = fmaf(k.ga, xh, k.be) > 0.f ? acc[r] : 0.f;
      s1 += (double)dy; s2 += (double)dy * (double)xh;
    }
}
// Batch-norm sums are collected in kHead2Groups copies (CTA c adds to copy c % kHead2Groups): the L2 serialises atomics per
// address, and 148 CTAs adding to one word cost 4 - 10 us per barrier (measured: arrival -> release); the leader adds the copies.
__device__ __forceinline__ double* grp_fwd(const Head2& h, int set) { return h.gsums[set] + (size_t)(blockIdx.x % kHead2Groups) * 2 * h.bn[set].C; }
__device__ __forceinline__ double* grp_bwd(const Head2& h, int set) { return h.gbsums[set] + (size_t)(blockIdx.x % kHead2Groups) * 2 * h.bn[set].C; }
__device__ __forceinline__ void add_sums(double* dst, int col, double a, double b) {
  if (a != 0.0 || b != 0.0) { atomicAdd(dst + 2 * col, a); atomicAdd(dst + 2 * col + 1, b); }
}

// ---- grid barrier with a leader section
struct Leader {
  int n_sync; int sync[2]; int bwd; int scalars;     // sets whose sums are complete at this barrier (and all-reduced over ranks)
  int fin_rows_n;                                    // forward: count = B*T (1) or B (0)
  int eval_stats;
};

// All-reduce of fp64 vectors over the ranks through the peer mailboxes, flag-in-data: every double travels as ONE 16-byte store
// {low, epoch, high, epoch} into the receiver's memory; the receiver polls the entry until both epoch words match (a torn
// 16-byte store is harmless: each half carries its own copy).  One NVLink trip per exchange; sums in rank order, so every rank
// gets bit-identical results.  A slot is reused one step later with a different epoch (head_dyn: one epoch per launch).
__device__ __forceinline__ void leader_p2p(const HeadDyn& d, int slot, double* const* buf, const int* n, int nbuf) {
  const int tid = threadIdx.x;
  int total = 0;
  for (int b = 0; b < nbuf; ++b) total += n[b];
  const uint32_t ep = d.p2p_epoch;
  for (int i = tid; i < total; i += kT2) {
    int b = 0, o = i;
    while (o >= n[b]) { o -= n[b]; ++b; }
    const unsigned long long bits = (unsigned long long)__double_as_longlong(buf[b][o]);
    const uint4 v = make_uint4((uint32_t)bits, ep, (uint32_t)(bits >> 32), ep);
    for (int p = 0; p < d.world; ++p) {
      uint4* dst = d.peer_ll[p] + (size_t)(slot * d.world + d.rank) * kP2PMaxDoubles + i;
      asm volatile("st.relaxed.sys.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    }
  }
  const uint4* mine = d.peer_ll[d.rank] + (size_t)slot * d.world * kP2PMaxDoubles;
  for (int i = tid; i < total; i += kT2) {
    double s = 0.0;
    for (int p = 0; p < d.world; ++p) {
      const uint4* src = mine + (size_t)p * kP2PMaxDoubles + i;
      uint4 v;
      uint32_t spins = 0;
      for (;;) {
        asm volatile("ld.relaxed.sys.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(src) : "memory");
        if (v.y == ep && v.w == ep) break;
        if (++spins > (1u << 22)) { *d.p2p_err = 1u + (uint32_t)slot; break; }
        __nanosleep(32);
      }
      s += __longlong_as_double((long long)(((unsigned long long)v.z << 32) | (unsigned long long)v.x));
    }
    int b = 0, o = i;
    while (o >= n[b]) { o -= n[b]; ++b; }
    buf[b][o] = s;
  }
  __syncthreads();
}

// sum of the kHead2Groups copies of element i of a set's sums (all loads in flight at once); the copies go back to zero
__device__ __forceinline__ double take_copies(double* g, int C, int i) {
  double v[kHead2Groups];
#pragma unroll
  for (int q = 0; q < kHead2Groups; ++q) v[q] = __ldcg(g + (size_t)q * 2 * C + i);
  double t = 0.0;
#pragma unroll
  for (int q = 0; q < kHead2Groups; ++q) { t += v[q]; g[(size_t)q * 2 * C + i] = 0.0; }
  return t;
}
__device__ __forceinline__ void bn_finalize_col(const BnSet& s, int c, double sum, double sq, double count, float mm, float mv) {
  // k_bn_finalize's arithmetic (kernels_head.cu)
  const double mean = sum / count;
  double var = sq / count - mean * mean;
  if (var < 0.0) var = 0.0;
  s.stat[2 * c] = (float)mean;
  s.stat[2 * c + 1] = (float)(1.0 / sqrt(var + (double)kBnEps));
  s.mmean[c] = mm - (mm - (float)mean) * kBnDecay;
  s.mvar[c] = mv - (mv - (float)var) * kBnDecay;
}
__device__ __noinline__ void leader_work(const Head2& h, const HeadDyn& d, const Leader& L, int barrier_index) {
  const int tid = threadIdx.x;
  if (!d.training) {
    if (L.eval_stats)
      for (int k = 0; k < BN_COUNT; ++k) {
        const BnSet& s = h.bn[k];
        for (int c = tid; c < s.C; c += kT2) { s.stat[2 * c] = s.mmean[c]; s.stat[2 * c + 1] = 1.0f / sqrtf(s.mvar[c] + kBnEps); }
      }
    return;
  }
  const float gs = 1.0f / (float)d.world;
  if (d.world == 1) {
    // one pass, one L2 round trip per thread: the copies of the column's two sums and its moving statistics are requested together
    for (int k = 0; k < L.n_sync; ++k) {
      const BnSet& s = h.bn[L.sync[k]];
      double* g = L.bwd ? h.gbsums[L.sync[k]] : h.gsums[L.sync[k]];
      const double count = L.fin_rows_n ? d.cntN : d.cntB;
      for (int c = tid; c < s.C; c += kT2) {
        float mm = 0.f, mv = 0.f;
        if (!L.bwd) { mm = __ldcg(s.mmean + c); mv = __ldcg(s.mvar + c); }
        const double a = take_copies(g, s.C, 2 * c), b = take_copies(g, s.C, 2 * c + 1);
        if (!L.bwd) bn_finalize_col(s, c, a, b, count, mm, mv);
        else {
          // gamma / beta gradients of the set; consumers read S1 / S2 from the canonical array
          s.bsums[2 * c] = a; s.bsums[2 * c + 1] = b;
          s.dbeta[c] += (float)a * gs;
          s.dgamma[c] += (float)b * gs;
        }
      }
    }
    return;
  }
  // data parallel: copies -> canonical array, all-reduce over the ranks (peer mailboxes), then finalize / parameter gradients
  for (int k = 0; k < L.n_sync; ++k) {
    const BnSet& s = h.bn[L.sync[k]];
    double* g = L.bwd ? h.gbsums[L.sync[k]] : h.gsums[L.sync[k]];
    double* dst = L.bwd ? s.bsums : s.sums;
    for (int i = tid; i < 2 * s.C; i += kT2) dst[i] = take_copies(g, s.C, i);
  }
  __syncthreads();
  if (L.n_sync > 0 || L.scalars) {
    double* buf[3]; int n[3]; int nb = 0;
    for (int k = 0; k < L.n_sync; ++k) { const BnSet& s = h.bn[L.sync[k]]; buf[nb] = L.bwd ? s.bsums : s.sums; n[nb++] = 2 * s.C; }
    if (L.scalars) { buf[nb] = h.dp_scalars; n[nb++] = 8; }
    leader_p2p(d, d.p2p_slot0 + barrier_index, buf, n, nb);
  }
  for (int k = 0; k < L.n_sync; ++k) {
    const BnSet& s = h.bn[L.sync[k]];
    if (!L.bwd) {
      const double count = L.fin_rows_n ? d.cntN : d.cntB;
      for (int c = tid; c < s.C; c += kT2) {
        bn_finalize_col(s, c, s.sums[2 * c], s.sums[2 * c + 1], count, s.mmean[c], s.mvar[c]);
        s.sums[2 * c] = 0.0;
        s.sums[2 * c + 1] = 0.0;
      }
    } else {
      for (int c = tid; c < s.C; c += kT2) {
        s.dbeta[c] += (float)s.bsums[2 * c] * gs;
        s.dgamma[c] += (float)s.bsums[2 * c + 1] * gs;
      }
    }
  }
}

// Weights of the NEXT phase, copied into shared memory by the threads that only wait at a barrier (thread 0 arrives / polls):
// the column kernel then reads its weights with conflict-free LDS instead of a chain of L2 round trips (the phases were bound
// by exactly that latency: 13 batches of 8 loads for a 100-long contraction).
struct Prefetch { const float* s0; int n0; const float* s1; int n1; };
__device__ __forceinline__ Prefetch no_prefetch() { return Prefetch{nullptr, 0, nullptr, 0}; }
__device__ __forceinline__ void copy_weights(float* __restrict__ wbuf, const Prefetch& pf, int t, int nt) {
  // t in [0, nt): this thread's index among the copying threads
#pragma unroll 1
  for (int part = 0; part < 2; ++part) {
    const float* __restrict__ src = part ? pf.s1 : pf.s0;
    const int n = part ? pf.n1 : pf.n0;
    float* dst = wbuf + (part ? pf.n0 : 0);
    for (int i0 = t; i0 < n; i0 += 16 * nt) {
      float v[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) v[u] = i0 + u * nt < n ? __ldg(src + i0 + u * nt) : 0.f;
#pragma unroll
      for (int u = 0; u < 16; ++u) if (i0 + u * nt < n) dst[i0 + u * nt] = v[u];
    }
  }
}

__device__ __forceinline__ void grid_barrier(const Head2& h, const HeadDyn& d, unsigned& epoch, const Leader& L, int& n_barrier,
                                             float* wbuf, const Prefetch& pf) {
  unsigned* bar = d.bar;
  __syncthreads();
  if (d.trace_cta != nullptr && threadIdx.x == 0 && n_barrier < 16 && blockIdx.x < 256) {
    unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); d.trace_cta[n_barrier * 256 + blockIdx.x] = t;
  }
  if (blockIdx.x == 0) {
    if (threadIdx.x == 0) {
      unsigned spins = 0;
      while (ld_relaxed_u32(bar) < gridDim.x - 1) {
        if (++spins > (1u << 26)) { bar[2] = 1u + (unsigned)n_barrier; break; }
      }
      fence_acq_rel_gpu();
    } else if (gridDim.x == 1) {
      copy_weights(wbuf, pf, threadIdx.x - 1, kT2 - 1);
    }
    __syncthreads();
    leader_work(h, d, L, n_barrier);
    __syncthreads();
    if (threadIdx.x == 0) {
      if (d.trace != nullptr && n_barrier < 29) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); d.trace[n_barrier] = t; }
      bar[0] = 0u;
      __threadfence();
      st_release_u32(bar + 32, epoch + 1u);
    }
  } else {
    if (threadIdx.x == 0) {
      __threadfence();
      atomicAdd(bar, 1u);
      unsigned spins = 0;
      while ((int)(ld_relaxed_u32(bar + 32) - (epoch + 1u)) < 0) {
        if (++spins > (1u << 24)) { bar[2] = 1000u + (unsigned)n_barrier; break; }
        __nanosleep(32);
      }
      fence_acq_rel_gpu();
    } else {
      copy_weights(wbuf, pf, threadIdx.x - 1, kT2 - 1);
    }
    __syncthreads();
  }
  epoch += 1u;
  ++n_barrier;
}
__device__ __forceinline__ Leader leader_of(int a, int b, int bwd, int rows_n, int scalars = 0) {
  Leader L;
  L.n_sync = (a >= 0) + (b >= 0); L.sync[0] = a; L.sync[1] = b; L.bwd = bwd; L.scalars = scalars; L.fin_rows_n = rows_n; L.eval_stats = 0;
  return L;
}

// ---- attention pooling weights of one sample (pamrec.py:272-282), one warp: a = softmax_t(mask ? relu(BN(z2)) : -(2^32)+1)
__device__ __forceinline__ void pool_weights_w(const float* __restrict__ Z2, const BnC& k, const int* __restrict__ mask, int64_t base,
                                               int T, int lane, float* aw) {
  float s[8];
  float m = -INFINITY;
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    const int t = jj * 32 + lane;
    float val = -INFINITY;
    if (t < T) {
      const float sv = bn_act(Z2[base + t], k);
      val = (mask[base + t] == 1) ? sv : kMaskNeg;
    }
    s[jj] = val;
    m = fmaxf(m, val);
  }
  m = warp_max(m);
  float sum = 0.f;
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    const int t = jj * 32 + lane;
    const float e = (t < T) ? expf(s[jj] - m) : 0.f;
    s[jj] = e;
    sum += e;
  }
  sum = warp_sum(sum);
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    const int t = jj * 32 + lane;
    if (t < T) aw[t] = s[jj] / sum;
  }
  __syncwarp();
}

// block-wide sum of a double (all kT2 threads call); sh: >= kT2 / 32 doubles
__device__ __forceinline__ double block_sum_d(double v, double* sh) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum_d(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  double r = 0.0;
#pragma unroll
  for (int k = 0; k < kT2 / 32; ++k) r += sh[k];
  return r;
}

// ---- L1 + L2 + L3 and their gradients (base_model.py:196-242, pamrec.py:70-106), spread as thinly as the arithmetic allows -
// the phase is a chain of transcendental functions per unit, so its duration is the LONGEST chain, not the sum:
//   * cross entropy (or the softmax loss): one (row, head) pair - or one (softmax group, head) pair - per lane;
//   * ApproxNDCG (restated from TensorFlow-Ranking 0.3.x, oracle/pamrec_oracle.py:approx_ndcg_loss): one listwise group per
//     8 lanes, lane i < 5 owns element i: its score, its rank (4 pairwise sigmoids), its gain / discount terms; the other
//     elements' values arrive by shuffles.
// nval = number of listwise groups with a non-zero label sum (over all ranks): dp_scalars[0], counted by the forward kernel.
__device__ __forceinline__ float sigm(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float xent(float x, float y) { return fmaxf(x, 0.f) - x * y + log1pf(expf(-fabsf(x))); }
__device__ __forceinline__ void loss_rows_item(const Head2& h, const HeadDyn& d, int item) {
  const int lane = threadIdx.x & 31, B = d.B;
  const float inv_b = 1.0f / (float)d.Bg;
  const int u = item * 32 + lane;
  double a0 = 0.0, a1 = 0.0;
  if (d.sm_group == 0) {
    const int b = u >> 1, head = u & 1;
    if (b < B) {
      const float x = h.logits[3 * b + head];
      const float y = head ? d.y_play[b] : d.y_sat[b];
      const double a = (double)xent(x, y);
      if (head) a1 = a; else a0 = a;
      h.d_logits[3 * b + head] = (head ? d.fuzhu_w : 1.0f) * (sigm(x) - y) * inv_b;
    }
  } else {
    // hparams.loss == "softmax":  -group * mean(log(where(y == 1, softmax, 1))) over all B elements; units are (group, head) pairs
    const int sm = d.sm_group;
    const float scale = (float)sm * inv_b;
    if (u < 2 * (B / sm)) {
      const int head = u & 1, r0 = (u >> 1) * sm;
      const float* y = head ? d.y_play : d.y_sat;
      float mx = -INFINITY;
      for (int i = 0; i < sm; ++i) mx = fmaxf(mx, h.logits[3 * (r0 + i) + head]);
      float se = 0.f;
      int n_pos = 0;
      for (int i = 0; i < sm; ++i) { se += expf(h.logits[3 * (r0 + i) + head] - mx); n_pos += y[r0 + i] == 1.0f; }
      const float lse = mx + logf(se), wgt = head ? d.fuzhu_w : 1.0f;
      double acc = 0.0;
      for (int i = 0; i < sm; ++i) {
        const float x = h.logits[3 * (r0 + i) + head];
        const bool pos = y[r0 + i] == 1.0f;
        if (pos) acc += (double)(lse - x);
        h.d_logits[3 * (r0 + i) + head] = wgt * scale * ((float)n_pos * expf(x - lse) - (pos ? 1.0f : 0.f));
      }
      if (head) a1 = acc * (double)sm; else a0 = acc * (double)sm;
    }
  }
  if (item == 0) {
    const int G = B / PAMREC_GROUP;
    for (int b = G * 5 + lane; b < B; b += 32) h.d_logits[3 * b + 2] = 0.f;    // rows outside a complete listwise group
  }
  a0 = warp_sum_d(a0); a1 = warp_sum_d(a1);
  if (lane == 0) {
    if (a0 != 0.0) atomicAdd(h.loss_acc, a0 / (double)d.Bg);
    if (a1 != 0.0) atomicAdd(h.loss_acc + 1, (double)d.fuzhu_w * a1 / (double)d.Bg);
  }
}
__device__ __forceinline__ void loss_ndcg_item(const Head2& h, const HeadDyn& d, int item) {
  const int lane = threadIdx.x & 31, sub = lane & 7, base = lane & ~7;
  const int G = d.B / PAMREC_GROUP;
  const int g = item * 4 + (lane >> 3);
  const bool on = g < G && sub < 5;
  const double nval = *h.dp_scalars;
  const float alpha = 10.0f;
  const int row = on ? g * 5 + sub : 0;
  const float s = on ? sigm(h.logits[3 * row + 2]) : 0.f;              // pamrec.py:74
  float y = on ? d.plays[row] : 0.f;
  float sj[5], yj[5];
#pragma unroll
  for (int j = 0; j < 5; ++j) { sj[j] = __shfl_sync(0xffffffffu, s, base + j); yj[j] = __shfl_sync(0xffffffffu, y, base + j); }
  const bool valid = (yj[0] + yj[1] + yj[2] + yj[3] + yj[4]) > 0.f;
  if (!valid) {
    y = 1e-10f;
#pragma unroll
    for (int j = 0; j < 5; ++j) yj[j] = 1e-10f;
  }
  const float gain = exp2f(y) - 1.0f;
  float rank = 1.0f, pq[5];                                           // 0.5 + sigmoid(0) of the pair (i, i)
  int pos = 0;                                                        // place of y in the descending order (ties: by index)
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    pq[j] = 0.f;
    if (j != sub) {
      const float p = sigm(alpha * (sj[j] - s));
      rank += p;
      pq[j] = p * (1.0f - p);
      pos += (yj[j] > y) || (yj[j] == y && j < sub);
    }
  }
  const float l1p = log1pf(rank);
  float dcg = on ? gain / l1p : 0.f, idcg = on ? gain / log1pf((float)(pos + 1)) : 0.f;
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) { dcg += __shfl_xor_sync(0xffffffffu, dcg, o); idcg += __shfl_xor_sync(0xffffffffu, idcg, o); }
  const float inv = idcg > 0.f ? 1.0f / idcg : 0.f;
  const float w = valid ? 1.0f : 0.f;
  const float coef = (nval > 0.0) ? d.order_w * w / (float)nval : 0.f;
  const float dLr = gain * inv / (l1p * l1p * (1.0f + rank));
  float acc = 0.f;                                                    // d loss / d s_i = alpha sum_{j != i} (dLr_j - dLr_i) p_ij (1 - p_ij)
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const float dj = __shfl_sync(0xffffffffu, dLr, base + j);
    acc += alpha * pq[j] * (dj - dLr);
  }
  if (on) h.d_logits[3 * row + 2] = coef * acc * s * (1.0f - s);
  double a2 = (on && sub == 0) ? (double)(w * -(dcg * inv)) : 0.0;
  a2 = warp_sum_d(a2);
  if (lane == 0 && a2 != 0.0 && nval > 0.0) atomicAdd(h.loss_acc + 2, (double)d.order_w * a2 / nval);
}

// samples of this CTA.  CTA 0 is the coordinator of the grid barriers (batch-norm finalize, data-parallel exchange): it owns no
// rows, so that the other CTAs never wait for its share of a phase on top of its leader work.
struct Rows { int b0, b1; };
__device__ __forceinline__ Rows my_rows(int B) {
  const int workers = max((int)gridDim.x - 1, 1);
  const int me = gridDim.x > 1 ? (int)blockIdx.x - 1 : 0;
  const int per = (B + workers - 1) / workers;
  Rows r;
  r.b0 = me < 0 ? B : min(B, me * per);
  r.b1 = me < 0 ? B : min(B, r.b0 + per);
  return r;
}

}  // namespace

// transposed weights in the workspace (written at the tail of the forward kernel): offsets in floats
constexpr int kWT_t1 = 0;                      // towers layer 1:  [3][64][100]   (n, k)
constexpr int kWT_t0 = kWT_t1 + 3 * 6400;      // towers layer 0:  [3][100][84]
constexpr int kWT_e1 = kWT_t0 + 3 * 8400;      // experts layer 1: [5][64][100]
constexpr int kWT_g1 = kWT_e1 + 5 * 6400;      // gates layer 1:   [2][5][64]
constexpr int kWT_x0 = kWT_g1 + 2 * 320;       // experts then gates layer 0 as ONE [628][40] matrix: rows g*100+n (expert g), 500+g*64+n (gate g)
constexpr int kWT_total = kWT_x0 + 628 * 40;
static_assert(kWT_total == kHead2WtFloats, "head2.h: workspace size of the transposed weights");
__device__ __forceinline__ void head2_transpose_weights(const Head2& h) {
  float* wT = h.wT;
  const int64_t gtid = (int64_t)blockIdx.x * kT2 + threadIdx.x, gsz = (int64_t)gridDim.x * kT2;
  for (int64_t i = gtid; i < kWT_total; i += gsz) {
    float v;
    if (i < kWT_t0) { const int j = (int)i, g = j / 6400, r = j % 6400, n = r / 100, k = r % 100; v = h.t_w1[g * 6400 + k * 64 + n]; }
    else if (i < kWT_e1) { const int j = (int)i - kWT_t0, g = j / 8400, r = j % 8400, n = r / 84, k = r % 84; v = h.t_w0[g * 8400 + k * 100 + n]; }
    else if (i < kWT_g1) { const int j = (int)i - kWT_e1, g = j / 6400, r = j % 6400, n = r / 100, k = r % 100; v = h.e_w1[g * 6400 + k * 64 + n]; }
    else if (i < kWT_x0) { const int j = (int)i - kWT_g1, g = j / 320, r = j % 320, n = r / 64, k = r % 64; v = h.g_w1[g * 320 + k * 5 + n]; }
    else {
      const int j = (int)i - kWT_x0, row = j / 40, k = j % 40;
      if (row < 500) { const int g = row / 100, n = row % 100; v = h.e_w0[g * 4000 + k * 100 + n]; }
      else { const int rr = row - 500, g = rr / 64, n = rr % 64; v = h.g_w0[g * 2560 + k * 64 + n]; }
    }
    wT[i] = v;
  }
}

// ================================================================================================ forward
__global__ void __launch_bounds__(kT2, 1) k_head2_fwd(const __grid_constant__ Head2 h, const __grid_constant__ HeadDyn d) {
  extern __shared__ __align__(16) float dsm[];
  float* wbuf = dsm;                                          // weights of the current / next phase
  float* xs = dsm + kWBuf;                                    // staged inputs of the current chunk, [column][row]
  __shared__ __align__(16) float w0s[kD * 20 + 64];           // score layer 0 weights [40][20], b0[20], w1[20], b1
  __shared__ double shd[64];
  __shared__ unsigned s_epoch;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0 && blockIdx.x == 0 && d.trace != nullptr) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); d.trace[31] = t; }
  if (tid == 0) s_epoch = ld_relaxed_u32(d.bar + 32);
  for (int i = tid; i < kD * 20; i += kT2) w0s[i] = h.s_w0[i];
  if (tid < 20) { w0s[800 + tid] = h.s_b0[tid]; w0s[820 + tid] = h.s_w1[tid]; }
  if (tid == 0) w0s[840] = h.s_b1[0];
  __syncthreads();
  unsigned epoch = s_epoch;
  int n_barrier = 0;
  const bool train = d.training != 0;
  const int T = d.T;
  const Rows R = my_rows(d.B);
  const int64_t tok0 = (int64_t)R.b0 * T, tok1 = (int64_t)R.b1 * T;
  // training: grid barrier (the waiting threads copy the next phase's weights); scoring: batch-norm statistics are constants, the
  // CTAs never meet again after the first barrier and every CTA copies its weights itself
  auto sync_point = [&](const Leader& L, const Prefetch& pf) {
    if (train) grid_barrier(h, d, epoch, L, n_barrier, wbuf, pf);
    else { __syncthreads(); copy_weights(wbuf, pf, tid, kT2); __syncthreads(); }
  };
  if (!train) { Leader L = leader_of(-1, -1, 0, 0); L.eval_stats = 1; grid_barrier(h, d, epoch, L, n_barrier, wbuf, no_prefetch()); }

  // ---- the coordinator counts the listwise groups with a non-zero label sum (ApproxNDCG weight, pamrec.py:76): dp_scalars[0];
  //      data parallel: summed over the ranks with the sums of the first barrier
  if (train && blockIdx.x == 0) {
    const int G = d.B / PAMREC_GROUP;
    double cnt = 0.0;
    for (int g = tid; g < G; g += kT2) {
      float sg = 0.f;
#pragma unroll
      for (int i = 0; i < PAMREC_GROUP; ++i) sg += d.plays[g * PAMREC_GROUP + i];
      cnt += (sg > 0.f) ? 1.0 : 0.0;
    }
    cnt = block_sum_d(cnt, shd);
    if (tid == 0) h.dp_scalars[0] = cnt;
  }
  // ---- F1: z1 = H W0 + b0 over the CTA's tokens in chunks of 125: the chunk's rows (20 KB, contiguous) go through shared memory,
  //          the next chunk's rows are already in flight while thread (slot, j) computes column j of tokens slot, slot + 25, ...
  {
    constexpr int kChunk = 5 * kSlots;
    const int slot = tid / 20, j = tid % 20;
    double s = 0.0, q = 0.0;
    float wc[kD];
#pragma unroll
    for (int k = 0; k < kD; ++k) wc[k] = w0s[k * 20 + (slot < kSlots ? j : 0)];
    const float b = w0s[800 + j];
    float4 pre[3];
    auto load_chunk = [&](int64_t c0) {
      const int nq = (int)min((int64_t)kChunk, tok1 - c0) * 10;
#pragma unroll
      for (int u = 0; u < 3; ++u) { const int i = tid + u * kT2; pre[u] = i < nq ? ld4(h.H + c0 * kD + 4 * i) : f4_zero(); }
    };
    if (tok0 < tok1) load_chunk(tok0);
    for (int64_t c0 = tok0; c0 < tok1; c0 += kChunk) {
      const int nt = (int)min((int64_t)kChunk, tok1 - c0);
      __syncthreads();
#pragma unroll
      for (int u = 0; u < 3; ++u) { const int i = tid + u * kT2; if (i < kChunk * 10) st4(xs + 4 * i, pre[u]); }
      __syncthreads();
      if (c0 + kChunk < tok1) load_chunk(c0 + kChunk);
      if (slot < kSlots) {
#pragma unroll
        for (int u = 0; u < 5; ++u) {
          const int tl = slot + u * kSlots;
          if (tl < nt) {
            const float* hr = xs + tl * kD;
            float z = b;
#pragma unroll
            for (int i = 0; i < 10; ++i) {
              const float4 x = ld4(hr + 4 * i);
              z = fmaf(x.x, wc[4 * i], z); z = fmaf(x.y, wc[4 * i + 1], z); z = fmaf(x.z, wc[4 * i + 2], z); z = fmaf(x.w, wc[4 * i + 3], z);
            }
            h.z1[(c0 + tl) * 20 + j] = z;
            s += (double)z; q += (double)z * (double)z;
          }
        }
      }
    }
    __syncthreads();
    if (train) {
      // the 25 slot-threads of a column: reduce through shared memory (xs is free here)
      double* red = reinterpret_cast<double*>(xs);            // [2][25][20]
      if (slot < kSlots) { red[slot * 20 + j] = s; red[500 + slot * 20 + j] = q; }
      __syncthreads();
      if (tid < 40) {
        const int which = tid / 20, c = tid % 20;
        double t = 0.0;
        for (int k = 0; k < kSlots; ++k) t += red[which * 500 + k * 20 + c];
        if (t != 0.0) atomicAdd(grp_fwd(h, BN_S0) + 2 * c + which, t);
      }
    }
    sync_point(leader_of(BN_S0, -1, 0, 1, 1), Prefetch{h.e_w0, 5 * 4000, h.g_w0, 2 * 2560});
  }
  // ---- F2: z2 = relu(bn(z1)) w1 + b1, one thread per token
  __syncthreads();
  {
    const BnSet& s0 = h.bn[BN_S0];
    double s = 0.0, q = 0.0;
    for (int64_t tok = tok0 + tid; tok < tok1; tok += kT2) {
      const float* zr = h.z1 + tok * 20;
      float z = w0s[840];
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const float4 x = ld4(zr + 4 * i);
        z = fmaf(bn_act(x.x, bn_c(s0, 4 * i)), w0s[820 + 4 * i], z);
        z = fmaf(bn_act(x.y, bn_c(s0, 4 * i + 1)), w0s[820 + 4 * i + 1], z);
        z = fmaf(bn_act(x.z, bn_c(s0, 4 * i + 2)), w0s[820 + 4 * i + 2], z);
        z = fmaf(bn_act(x.w, bn_c(s0, 4 * i + 3)), w0s[820 + 4 * i + 3], z);
      }
      h.z2[tok] = z;
      s += (double)z; q += (double)z * (double)z;
    }
    if (train) {
      s = block_sum_d(s, shd); q = block_sum_d(q, shd);
      if (tid == 0 && (s != 0.0 || q != 0.0)) { atomicAdd(grp_fwd(h, BN_S1), s); atomicAdd(grp_fwd(h, BN_S1) + 1, q); }
    }
    sync_point(leader_of(BN_S1, -1, 0, 1), no_prefetch());
  }
  // ---- F3: pooling (warp per sample) -> new_long, then experts / gates layer 0 on the CTA's rows
  __syncthreads();
  {
    const BnC k1 = bn_c(h.bn[BN_S1], 0);
    float* aws = xs;                                          // [16 warps][256]
    for (int b = R.b0 + warp; b < R.b1; b += kT2 / 32) {
      const int64_t base = (int64_t)b * T;
      float* aw = aws + warp * PAMREC_MAX_T;
      pool_weights_w(h.z2, k1, d.mask, base, T, lane, aw);
      const int tg = lane / 10, c = lane % 10;
      float4 acc = f4_zero();
      if (lane < 30)
        for (int t = tg; t < T; t += 3) f4_fma(acc, aw[t], ld4(h.H + (base + t) * kD + 4 * c));
      const float4 a1 = f4_shfl_down(acc, 10), a2 = f4_shfl_down(acc, 20);
      if (lane < 10) {
        acc.x += a1.x + a2.x; acc.y += a1.y + a2.y; acc.z += a1.z + a2.z; acc.w += a1.w + a2.w;
        st4(h.new_long + (int64_t)b * kD + 4 * c, acc);
      }
      if (train || d.keep_aw) for (int t = lane; t < T; t += 32) h.aw[base + t] = aw[t];   // kept for the backward pass / pamrec_attention
      __syncwarp();
    }
    __syncthreads();
    double s[2] = {0.0, 0.0}, q[2] = {0.0, 0.0};
    for (int row0 = R.b0; row0 < R.b1; row0 += kRC) {
      const int nr = min(kRC, R.b1 - row0);
      __syncthreads();
      stage_cols(xs, 0, h.new_long, kD, kD, row0, nr, [](int, const float (&v)[kRC], float (&o)[kRC]) {
#pragma unroll
        for (int r = 0; r < kRC; ++r) o[r] = v[r];
      });
      __syncthreads();
#pragma unroll
      for (int pass = 0; pass < 2; ++pass) {
        const int col = tid + pass * kT2;                     // 0..499 expert columns, 500..627 gate columns
        if (col >= 628) continue;
        float acc[kRC];
        if (col < 500) {
          const int g = col / 100, n = col % 100;
          acc_set(acc, h.e_b0[g * 100 + n]);
          col_gemm(xs, 0, kD, wbuf + g * 4000 + n, 100, acc);
          epi_fwd(acc, h.ze0, 500, col, row0, nr, s[pass], q[pass]);
        } else {
          const int cg = col - 500, g = cg / 64, n = cg % 64;
          acc_set(acc, h.g_b0[g * 64 + n]);
          col_gemm(xs, 0, kD, wbuf + 20000 + g * 2560 + n, 64, acc);
          epi_fwd(acc, h.zg0, 128, cg, row0, nr, s[pass], q[pass]);
        }
      }
    }
    if (train) {
#pragma unroll
      for (int pass = 0; pass < 2; ++pass) {
        const int col = tid + pass * kT2;
        if (col < 500) add_sums(grp_fwd(h, BN_E0), col, s[pass], q[pass]);
        else if (col < 628) add_sums(grp_fwd(h, BN_G0), col - 500, s[pass], q[pass]);
      }
    }
    sync_point(leader_of(BN_E0, BN_G0, 0, 0), Prefetch{h.e_w1, 5 * 6400, h.g_w1, 2 * 320});
  }
  // ---- F4: experts / gates layer 1
  {
    double s = 0.0, q = 0.0;
    for (int row0 = R.b0; row0 < R.b1; row0 += kRC) {
      const int nr = min(kRC, R.b1 - row0);
      __syncthreads();
      stage_act(xs, 0, h.ze0, 500, 500, row0, nr, h.bn[BN_E0]);
      stage_act(xs, 500, h.zg0, 128, 128, row0, nr, h.bn[BN_G0]);
      __syncthreads();
      const int col = tid;                                    // 0..319 expert columns, 320..329 gate columns
      float acc[kRC];
      if (col < 320) {
        const int g = col / 64, n = col % 64;
        acc_set(acc, h.e_b1[g * 64 + n]);
        col_gemm(xs, g * 100, 100, wbuf + g * 6400 + n, 64, acc);
        epi_fwd(acc, h.ze1, 320, col, row0, nr, s, q);
      } else if (col < 330) {
        const int cg = col - 320, g = cg / 5, n = cg % 5;
        acc_set(acc, h.g_b1[g * 5 + n]);
        col_gemm(xs, 500 + g * 64, 64, wbuf + 32000 + g * 320 + n, 5, acc);
        epi_fwd(acc, h.zg1, 10, cg, row0, nr, s, q);
      }
    }
    if (train) {
      if (tid < 320) add_sums(grp_fwd(h, BN_E1), tid, s, q);
      else if (tid < 330) add_sums(grp_fwd(h, BN_G1), tid - 320, s, q);
    }
    sync_point(leader_of(BN_E1, BN_G1, 0, 0), Prefetch{h.t_w0, 3 * 8400, nullptr, 0});
  }
  // ---- F5: MMoE mixing (pamrec.py:46-50, 315-316) -> u = [main | tgt | sub | tgt]; towers layer 0
  {
    double s = 0.0, q = 0.0;
    float* es = xs + 168 * kRC;                               // relu(bn(ze1)) [320][8], then relu(bn(zg1)) [10][8]
    for (int row0 = R.b0; row0 < R.b1; row0 += kRC) {
      const int nr = min(kRC, R.b1 - row0);
      __syncthreads();
      stage_act(es, 0, h.ze1, 320, 320, row0, nr, h.bn[BN_E1]);
      stage_act(es, 320, h.zg1, 10, 10, row0, nr, h.bn[BN_G1]);
      __syncthreads();
      if (tid < 168) {
        const int c = tid;
        float o[kRC];
        if (c < 64 || (c >= 84 && c < 148)) {
          const int cc = c < 64 ? c : c - 84, gb = c < 64 ? 0 : 5;
#pragma unroll
          for (int r = 0; r < kRC; ++r) {
            float m = 0.f;
#pragma unroll
            for (int j = 0; j < 5; ++j) m = fmaf(es[(320 + gb + j) * kRC + r], es[(j * 64 + cc) * kRC + r], m);
            o[r] = m;
          }
        } else {
          const int cc = c < 84 ? c - 64 : c - 148;
#pragma unroll
          for (int r = 0; r < kRC; ++r) o[r] = r < nr ? h.tgt[(int64_t)(row0 + r) * kE + cc] : 0.f;
        }
#pragma unroll
        for (int r = 0; r < kRC; ++r) {
          if (r >= nr) o[r] = 0.f; else h.u[(int64_t)(row0 + r) * 168 + c] = o[r];
        }
        st4(xs + c * kRC, make_float4(o[0], o[1], o[2], o[3]));
        st4(xs + c * kRC + 4, make_float4(o[4], o[5], o[6], o[7]));
      }
      __syncthreads();
      if (tid < 300) {
        const int g = tid / 100, n = tid % 100;
        float acc[kRC];
        acc_set(acc, h.t_b0[g * 100 + n]);
        col_gemm(xs, g == 1 ? 84 : 0, 84, wbuf + g * 8400 + n, 100, acc);
        epi_fwd(acc, h.zt0, 300, tid, row0, nr, s, q);
      }
    }
    if (train && tid < 300) add_sums(grp_fwd(h, BN_T0), tid, s, q);
    sync_point(leader_of(BN_T0, -1, 0, 0), Prefetch{h.t_w1, 3 * 6400, nullptr, 0});
  }
  // ---- F6: towers layer 1
  {
    double s = 0.0, q = 0.0;
    for (int row0 = R.b0; row0 < R.b1; row0 += kRC) {
      const int nr = min(kRC, R.b1 - row0);
      __syncthreads();
      stage_act(xs, 0, h.zt0, 300, 300, row0, nr, h.bn[BN_T0]);
      __syncthreads();
      if (tid < 192) {
        const int g = tid / 64, n = tid % 64;
        float acc[kRC];
        acc_set(acc, h.t_b1[g * 64 + n]);
        col_gemm(xs, g * 100, 100, wbuf + g * 6400 + n, 64, acc);
        epi_fwd(acc, h.zt1, 192, tid, row0, nr, s, q);
      }
    }
    if (train && tid < 192) add_sums(grp_fwd(h, BN_T1), tid, s, q);
    sync_point(leader_of(BN_T1, -1, 0, 0), no_prefetch());
  }
  // ---- F7: logits (pamrec.py:212-215, 71); scoring: pred = sigmoid(logit 0)
  {
    for (int row0 = R.b0; row0 < R.b1; row0 += kRC) {
      const int nr = min(kRC, R.b1 - row0);
      __syncthreads();
      stage_act(xs, 0, h.zt1, 192, 192, row0, nr, h.bn[BN_T1]);
      __syncthreads();
      if (tid < 3 * kRC) {
        const int g = tid / kRC, r = tid % kRC;
        if (r < nr) {
          float z = h.t_bo[g];
          for (int k = 0; k < 64; ++k) z = fmaf(xs[(g * 64 + k) * kRC + r], h.t_wo[g * 64 + k], z);
          h.logits[(int64_t)(row0 + r) * 3 + g] = z;
          if (g == 0 && d.pred != nullptr) d.pred[row0 + r] = sigm(z);
        }
      }
    }
  }
  if (tid == 0 && blockIdx.x == 0 && d.trace != nullptr) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); d.trace[30] = t; d.trace[29] = (unsigned long long)n_barrier; }
  // ---- training: transposed weights for the dX chain of the backward kernel (nobody waits for this tail)
  if (train) head2_transpose_weights(h);
}

// ================================================================================================ backward (dX chain)
__global__ void __launch_bounds__(kT2, 1) k_head2_bwd(const __grid_constant__ Head2 h, const __grid_constant__ HeadDyn d) {
  extern __shared__ __align__(16) float dsm[];
  float* wbuf = dsm;                                          // transposed weights of the current / next phase
  float* xs = dsm + kWBuf;
  float* aux = xs + kXS * kRC;                                // [4096] combine / pooling / score scratch
  __shared__ double shd[64];
  __shared__ unsigned s_epoch;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0 && blockIdx.x == 0 && d.trace != nullptr) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); d.trace[31] = t; }
  if (tid == 0) s_epoch = ld_relaxed_u32(d.bar + 32);
  __syncthreads();
  unsigned epoch = s_epoch;
  int n_barrier = 0;
  const int T = d.T;
  const Rows R = my_rows(d.B);
  const int64_t tok0 = (int64_t)R.b0 * T, tok1 = (int64_t)R.b1 * T;
  const float* wT = h.wT;

  // ---- K0: the losses and d_logits, one warp per 32 listwise groups
  {
    const int G = d.B / PAMREC_GROUP;
    const int n_ndcg = (G + 3) / 4;
    const int n_units = d.sm_group > 0 ? 2 * (d.B / d.sm_group) : 2 * d.B;
    const int n_rows = max((n_units + 31) / 32, 1);
    const int workers = max((int)gridDim.x - 1, 1), me = gridDim.x > 1 ? (int)blockIdx.x - 1 : 0;
    if (d.B > 0 && me >= 0)
      for (int i = me + workers * warp; i < n_ndcg + n_rows; i += workers * (kT2 / 32)) {
        if (i < n_ndcg) loss_ndcg_item(h, d, i); else loss_rows_item(h, d, i - n_ndcg);
      }
    grid_barrier(h, d, epoch, leader_of(-1, -1, 1, 0), n_barrier, wbuf, Prefetch{wT + kWT_t1, 3 * 6400, nullptr, 0});
  }
  // ---- K1: dA(t1) = d_logits (x) w_out, sums of BN_T1
  {
    double s1 = 0.0, s2 = 0.0;
    if (tid < 192) {
      const int g = tid / 64, n = tid % 64;
      const float w = h.t_wo[g * 64 + n];
      const BnC k = bn_c(h.bn[BN_T1], tid);
      for (int b = R.b0; b < R.b1; ++b) {
        const int64_t i = (int64_t)b * 192 + tid;
        const float da = h.d_logits[(int64_t)b * 3 + g] * w;
        h.d_t1[i] = da;
        const float xh = (h.zt1[i] - k.mean) * k.inv;
        const float dy = fmaf(k.ga, xh, k.be) > 0.f ? da : 0.f;
        s1 += (double)dy; s2 += (double)dy * (double)xh;
      }
      add_sums(grp_bwd(h, BN_T1), tid, s1, s2);
    }
    grid_barrier(h, d, epoch, leader_of(BN_T1, -1, 1, 0), n_barrier, wbuf, no_prefetch());
  }
  // ---- K2: dz(t1) -> dA(t0) = dz(t1) W1^T, sums of BN_T0
  {
    double s1 = 0.0, s2 = 0.0;
    const BnC k = tid < 300 ? bn_c(h.bn[BN_T0], tid) : BnC{0.f, 0.f, 0.f, 0.f};
    for (int row0 = R.b0; row0 < R.b1; row0 += kRC) {
      const int nr = min(kRC, R.b1 - row0);
      __syncthreads();
      stage_dz(xs, 0, h.d_t1, h.zt1, 192, 192, row0, nr, h.bn[BN_T1], d.cntB);
      __syncthreads();
      if (tid < 300) {
        const int g = tid / 100, kk = tid % 100;
        float acc[kRC];
        acc_set(acc, 0.f);
        col_gemm(xs, g * 64, 64, wbuf + g * 6400 + kk, 100, acc);
        epi_bwd(acc, h.d_t0, h.zt0, 300, tid, row0, nr, k, s1, s2);
      }
    }
    if (tid < 300) add_sums(grp_bwd(h, BN_T0), tid, s1, s2);
    grid_barrier(h, d, epoch, leader_of(BN_T0, -1, 1, 0), n_barrier, wbuf, Prefetch{wT + kWT_t0, 3 * 8400, nullptr, 0});
  }
  // ---- K3: dz(t0) -> d_u = dz(t0) W0^T -> mixing backward: dA(e1), dA(g1), d_tgt; sums of BN_E1 / BN_G1
  {
    double s1 = 0.0, s2 = 0.0;                                // tid < 320: expert column tid; 320..399: gate column (tid - 320) / 8, row (tid - 320) % 8
    const BnC k = tid < 320 ? bn_c(h.bn[BN_E1], tid) : BnC{0.f, 0.f, 0.f, 0.f};
    const BnC kg = (tid >= 320 && tid < 400) ? bn_c(h.bn[BN_G1], (tid - 320) >> 3) : BnC{0.f, 0.f, 0.f, 0.f};
    float* du = aux;                                          // [168][8]
    float* gt = aux + 168 * kRC;                              // relu(bn(zg1)) [10][8]
    for (int row0 = R.b0; row0 < R.b1; row0 += kRC) {
      const int nr = min(kRC, R.b1 - row0);
      __syncthreads();
      stage_dz(xs, 0, h.d_t0, h.zt0, 300, 300, row0, nr, h.bn[BN_T0], d.cntB);
      stage_act(gt, 0, h.zg1, 10, 10, row0, nr, h.bn[BN_G1]);
      stage_act(xs, 300, h.ze1, 320, 320, row0, nr, h.bn[BN_E1]);      // e = relu(bn(ze1)) for the gate gradients
      __syncthreads();
      if (tid < 168) {
        float acc[kRC];
        acc_set(acc, 0.f);
        if (tid < 84) {
          col_gemm(xs, 0, 100, wbuf + tid, 84, acc);
          col_gemm(xs, 200, 100, wbuf + 2 * 8400 + tid, 84, acc);
        } else {
          col_gemm(xs, 100, 100, wbuf + 8400 + (tid - 84), 84, acc);
        }
        st4(du + tid * kRC, make_float4(acc[0], acc[1], acc[2], acc[3]));
        st4(du + tid * kRC + 4, make_float4(acc[4], acc[5], acc[6], acc[7]));
      }
      __syncthreads();
      // d_tgt = d_u[64:84] + d_u[148:168]
      if (tid >= 480 && tid < 500) {
        const int c = tid - 480;
        for (int r = 0; r < nr; ++r) h.d_tgt[(int64_t)(row0 + r) * kE + c] = du[(64 + c) * kRC + r] + du[(148 + c) * kRC + r];
      }
      if (tid < 320) {
        // dA(e1)[j][c] = g_main[j] d_main[c] + g_sub[j] d_sub[c]
        const int j = tid / 64, c = tid % 64;
#pragma unroll
        for (int r = 0; r < kRC; ++r)
          if (r < nr) {
            const int64_t i = (int64_t)(row0 + r) * 320 + tid;
            const float da = gt[j * kRC + r] * du[c * kRC + r] + gt[(5 + j) * kRC + r] * du[(84 + c) * kRC + r];
            h.d_e1[i] = da;
            const float xh = (h.ze1[i] - k.mean) * k.inv;
            const float dy = fmaf(k.ga, xh, k.be) > 0.f ? da : 0.f;
            s1 += (double)dy; s2 += (double)dy * (double)xh;
          }
      } else if (tid < 400) {
        // dA(g1)[jj] = sum_c e[j][c] d_{main|sub}[c]: thread (jj, r)
        const int jj = (tid - 320) >> 3, r = (tid - 320) & 7, j = jj % 5, off = jj < 5 ? 0 : 84;
        if (r < nr) {
          float da = 0.f;
          for (int c = 0; c < 64; ++c) da = fmaf(xs[(300 + j * 64 + c) * kRC + r], du[(off + c) * kRC + r], da);
          const int64_t i = (int64_t)(row0 + r) * 10 + jj;
          h.d_g1[i] = da;
          const float xh = (h.zg1[i] - kg.mean) * kg.inv;
          const float dy = fmaf(kg.ga, xh, kg.be) > 0.f ? da : 0.f;
          s1 += (double)dy; s2 += (double)dy * (double)xh;
        }
      }
    }
    if (tid < 320) add_sums(grp_bwd(h, BN_E1), tid, s1, s2);
    else if (tid < 400) add_sums(grp_bwd(h, BN_G1), (tid - 320) >> 3, s1, s2);
    grid_barrier(h, d, epoch, leader_of(BN_E1, BN_G1, 1, 0), n_barrier, wbuf, Prefetch{wT + kWT_e1, 5 * 6400 + 2 * 320, nullptr, 0});
  }
  // ---- K4: dz(e1), dz(g1) -> dA(e0), dA(g0); sums of BN_E0 / BN_G0
  {
    double s1[2] = {0.0, 0.0}, s2[2] = {0.0, 0.0};
    BnC kc[2];
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int col = tid + pass * kT2;
      kc[pass] = col < 500 ? bn_c(h.bn[BN_E0], col) : (col < 628 ? bn_c(h.bn[BN_G0], col - 500) : BnC{0.f, 0.f, 0.f, 0.f});
    }
    for (int row0 = R.b0; row0 < R.b1; row0 += kRC) {
      const int nr = min(kRC, R.b1 - row0);
      __syncthreads();
      stage_dz(xs, 0, h.d_e1, h.ze1, 320, 320, row0, nr, h.bn[BN_E1], d.cntB);
      stage_dz(xs, 320, h.d_g1, h.zg1, 10, 10, row0, nr, h.bn[BN_G1], d.cntB);
      __syncthreads();
#pragma unroll
      for (int pass = 0; pass < 2; ++pass) {
        const int col = tid + pass * kT2;
        if (col >= 628) continue;
        float acc[kRC];
        acc_set(acc, 0.f);
        if (col < 500) {
          const int g = col / 100, kk = col % 100;
          col_gemm(xs, g * 64, 64, wbuf + g * 6400 + kk, 100, acc);
          epi_bwd(acc, h.d_e0, h.ze0, 500, col, row0, nr, kc[pass], s1[pass], s2[pass]);
        } else {
          const int cg = col - 500, g = cg / 64, kk = cg % 64;
          col_gemm(xs, 320 + g * 5, 5, wbuf + 32000 + g * 320 + kk, 64, acc);
          epi_bwd(acc, h.d_g0, h.zg0, 128, cg, row0, nr, kc[pass], s1[pass], s2[pass]);
        }
      }
    }
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int col = tid + pass * kT2;
      if (col < 500) add_sums(grp_bwd(h, BN_E0), col, s1[pass], s2[pass]);
      else if (col < 628) add_sums(grp_bwd(h, BN_G0), col - 500, s1[pass], s2[pass]);
    }
    grid_barrier(h, d, epoch, leader_of(BN_E0, BN_G0, 1, 0), n_barrier, wbuf, Prefetch{wT + kWT_x0, 628 * 40, nullptr, 0});
  }
  // ---- K5: dz(e0), dz(g0) -> d_new_long = [dz(e0) | dz(g0)] [W_e0 | W_g0]^T (one 628-long contraction split over 12 thread
  //          groups); pooling backward (warp per sample): dA(z2), sums of BN_S1
  {
    const BnC k1 = bn_c(h.bn[BN_S1], 0);
    double b1 = 0.0, b2 = 0.0;
    float* part = aux;                                        // [12][40][8] partial sums
    float* dnl = xs;                                          // d_new_long of the chunk [8][40] (the staged inputs are dead by then)
    for (int row0 = R.b0; row0 < R.b1; row0 += kRC) {
      const int nr = min(kRC, R.b1 - row0);
      __syncthreads();
      stage_dz(xs, 0, h.d_e0, h.ze0, 500, 500, row0, nr, h.bn[BN_E0], d.cntB);
      stage_dz(xs, 500, h.d_g0, h.zg0, 128, 128, row0, nr, h.bn[BN_G0], d.cntB);
      __syncthreads();
      if (tid < 480) {
        const int grp = tid / 40, c = tid % 40;               // 12 groups x 53 rows of the [628][40] transposed matrix (the last: 45)
        const int k0 = grp * 53, kn = min(53, 628 - k0);
        float acc[kRC];
        acc_set(acc, 0.f);
        col_gemm(xs, k0, kn, wbuf + k0 * 40 + c, 40, acc);
        float* p = part + (grp * 40 + c) * kRC;
        st4(p, make_float4(acc[0], acc[1], acc[2], acc[3]));
        st4(p + 4, make_float4(acc[4], acc[5], acc[6], acc[7]));
      }
      __syncthreads();
      if (tid < 40 * kRC) {
        const int r = tid / 40, c = tid % 40;
        float v = 0.f;
#pragma unroll
        for (int g = 0; g < 12; ++g) v += part[(g * 40 + c) * kRC + r];
        dnl[r * 40 + c] = v;
        if (r < nr) h.d_new_long[(int64_t)(row0 + r) * kD + c] = v;
      }
      __syncthreads();
      if (warp < nr) {
        const int b = row0 + warp;
        const int64_t base = (int64_t)b * T;
        float4 dn[10];
#pragma unroll
        for (int i = 0; i < 10; ++i) dn[i] = ld4(dnl + warp * 40 + 4 * i);
        float da[8], a[8];
        float dot = 0.f;
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const int t = jj * 32 + lane;
          float v = 0.f, av = 0.f;
          if (t < T) {
            const float* hr = h.H + (base + t) * kD;
#pragma unroll
            for (int i = 0; i < 10; ++i) v += f4_dot(dn[i], ld4(hr + 4 * i));
            av = h.aw[base + t];
            dot = fmaf(av, v, dot);
          }
          da[jj] = v; a[jj] = av;
        }
        dot = warp_sum(dot);
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
          const int t = jj * 32 + lane;
          if (t < T) {
            const float dv = (d.mask[base + t] == 1) ? a[jj] * (da[jj] - dot) : 0.f;
            h.d_z2[base + t] = dv;
            const float xh = (h.z2[base + t] - k1.mean) * k1.inv;
            const float dy = fmaf(k1.ga, xh, k1.be) > 0.f ? dv : 0.f;
            b1 += (double)dy; b2 += (double)dy * (double)xh;
          }
        }
      }
    }
    b1 = block_sum_d(b1, shd); b2 = block_sum_d(b2, shd);
    if (tid == 0 && (b1 != 0.0 || b2 != 0.0)) { atomicAdd(grp_bwd(h, BN_S1), b1); atomicAdd(grp_bwd(h, BN_S1) + 1, b2); }
    grid_barrier(h, d, epoch, leader_of(BN_S1, -1, 1, 1), n_barrier, wbuf, no_prefetch());
  }
  // score MLP constants in shared memory: W0 [40][20], its transpose, w1, BN coefficients
  float* w0s = aux;                                           // [800]  W0[k][j]
  float* w0t = aux + 800;                                     // [800]  W0^T[j][k]
  float* w1s = aux + 1600;                                    // [20]
  float* c0 = aux + 1620;                                     // BN_S0 backward coefficients [20][6]
  __syncthreads();
  for (int i = tid; i < 800; i += kT2) { const float v = h.s_w0[i]; w0s[i] = v; w0t[(i % 20) * 40 + i / 20] = v; }
  if (tid < 20) w1s[tid] = h.s_w1[tid];
  // ---- K6: dz2 -> dA(z1) = dz2 w1; sums of BN_S0; gradients of the score layer 1 (w1, b1); thread (slot, j)
  {
    const BnB k1 = bn_b(h.bn[BN_S1], 0, d.cntN);
    const int slot = tid / 20, j = tid % 20;
    double s1 = 0.0, s2 = 0.0, gw = 0.0, gb = 0.0;
    __syncthreads();
    if (slot < kSlots) {
      const BnC k0 = bn_c(h.bn[BN_S0], j);
      const float w1j = w1s[j];
      for (int64_t tok = tok0 + slot; tok < tok1; tok += kSlots) {
        const float dz2 = bn_dz(h.d_z2[tok], h.z2[tok], k1);
        const float xh = (h.z1[tok * 20 + j] - k0.mean) * k0.inv;
        const float y = fmaf(k0.ga, xh, k0.be);
        gw += (double)(fmaxf(y, 0.f) * dz2);
        if (j == 0) gb += (double)dz2;
        const float dy = y > 0.f ? dz2 * w1j : 0.f;
        s1 += (double)dy; s2 += (double)dy * (double)xh;
      }
    }
    double* red = reinterpret_cast<double*>(xs);              // [4][25][20]
    __syncthreads();
    if (slot < kSlots) { red[slot * 20 + j] = s1; red[500 + slot * 20 + j] = s2; red[1000 + slot * 20 + j] = gw; red[1500 + slot * 20 + j] = gb; }
    __syncthreads();
    if (tid < 80) {
      const int which = tid / 20, c = tid % 20;
      double t = 0.0;
      for (int k = 0; k < kSlots; ++k) t += red[which * 500 + k * 20 + c];
      if (t != 0.0) {
        if (which < 2) atomicAdd(grp_bwd(h, BN_S0) + 2 * c + which, t);
        else if (which == 2) atomicAdd(h.ds_w1 + c, (float)t);
        else if (c == 0) atomicAdd(h.ds_b1, (float)t);
      }
    }
    grid_barrier(h, d, epoch, leader_of(BN_S0, -1, 1, 1), n_barrier, wbuf, no_prefetch());
  }
  // ---- K7: dz1 -> dH = a_t d_new_long + dz1 W0^T  (the gradient of the encoder output, g_a);  dW0 = H^T dz1, db0.
  //          Batches of 50 tokens; everything a batch reads from global memory is requested one batch ahead:
  //          thread (token, k quad), tid < 500: its float4 of H, the token's pooling weight and its float4 of d_new_long;
  //          thread (slot, j), tid < 500: d_z2, z2, z1 of tokens slot and slot + 25.
  {
    constexpr int kTB = 2 * kSlots;
    const BnB k1 = bn_b(h.bn[BN_S1], 0, d.cntN);
    const int slot = tid / 20, j = tid % 20;
    const int sl_h = tid / 10, kq = tid % 10;
    if (tid < 20) {
      const BnB k = bn_b(h.bn[BN_S0], tid, d.cntN);
      c0[6 * tid] = k.mean; c0[6 * tid + 1] = k.inv; c0[6 * tid + 2] = k.ga; c0[6 * tid + 3] = k.be; c0[6 * tid + 4] = k.s1n; c0[6 * tid + 5] = k.s2n;
    }
    float* Hs = xs;                                           // [50][40] encoder outputs of the batch
    float* dzs = xs + kTB * kD;                               // [50][20] dz1 of the batch
    float gw[4] = {0.f, 0.f, 0.f, 0.f};                       // dW0[k][4 jq .. 4 jq + 3] of threads 0..199
    double gb = 0.0;
    const int wk = tid / 5, wjq = tid % 5;
    __syncthreads();
    const bool colthr = slot < kSlots;
    const BnB k0 = colthr ? BnB{c0[6 * j], c0[6 * j + 1], c0[6 * j + 2], c0[6 * j + 3], c0[6 * j + 4], c0[6 * j + 5]} : BnB{0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const float w1j = colthr ? w1s[j] : 0.f;
    float4 pH = f4_zero(), pDn = f4_zero();
    float pA = 0.f, pdA[2] = {0.f, 0.f}, pz2[2] = {0.f, 0.f}, pz1[2] = {0.f, 0.f};
    auto prefetch = [&](int64_t tb) {
      const int nt = (int)min((int64_t)kTB, tok1 - tb);
      if (tid < kTB * 10) {
        const bool ok = sl_h < nt;
        const int64_t tok = tb + sl_h;
        pH = ok ? ld4(h.H + tok * kD + 4 * kq) : f4_zero();
        pA = ok ? h.aw[tok] : 0.f;
        pDn = ok ? ld4(h.d_new_long + (tok / T) * kD + 4 * kq) : f4_zero();
      }
      if (colthr) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int sl = slot + u * kSlots;
          const int64_t tok = tb + sl;
          pdA[u] = sl < nt ? h.d_z2[tok] : 0.f; pz2[u] = sl < nt ? h.z2[tok] : 0.f; pz1[u] = sl < nt ? h.z1[tok * 20 + j] : 0.f;
        }
      }
    };
    if (tok0 < tok1) prefetch(tok0);
    for (int64_t tb = tok0; tb < tok1; tb += kTB) {
      const int nt = (int)min((int64_t)kTB, tok1 - tb);
      __syncthreads();                                        // the previous batch has been consumed
      float4 dn = pDn;
      const float a = pA;
      if (tid < kTB * 10) st4(Hs + 4 * tid, pH);
      if (colthr) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int sl = slot + u * kSlots;
          float dz1 = 0.f;
          if (sl < nt) {
            const float dz2 = bn_dz(pdA[u], pz2[u], k1);
            dz1 = bn_dz(dz2 * w1j, pz1[u], k0);
            gb += (double)dz1;
          }
          dzs[sl * 20 + j] = dz1;
        }
      }
      __syncthreads();
      if (tb + kTB < tok1) prefetch(tb + kTB);
      if (tid < kTB * 10 && sl_h < nt) {
        // dH[token][4 kq .. 4 kq + 3]
        float4 o = make_float4(a * dn.x, a * dn.y, a * dn.z, a * dn.w);
#pragma unroll
        for (int jj = 0; jj < 20; ++jj) f4_fma(o, dzs[sl_h * 20 + jj], ld4(w0t + jj * 40 + 4 * kq));
        st4(h.g_a + (tb + sl_h) * kD + 4 * kq, o);
      }
      if (tid < 200) {
        // dW0[k][4 jq ..] += sum over the batch's tokens
        float4 acc = make_float4(gw[0], gw[1], gw[2], gw[3]);
#pragma unroll 5
        for (int sl = 0; sl < nt; ++sl) f4_fma(acc, Hs[sl * 40 + wk], ld4(dzs + sl * 20 + 4 * wjq));
        gw[0] = acc.x; gw[1] = acc.y; gw[2] = acc.z; gw[3] = acc.w;
      }
    }
    if (tid < 200) {
#pragma unroll
      for (int i = 0; i < 4; ++i) if (gw[i] != 0.f) atomicAdd(h.ds_w0 + wk * 20 + 4 * wjq + i, gw[i]);
    }
    double* red = reinterpret_cast<double*>(aux + 2048);      // [25][20]
    __syncthreads();
    if (colthr) red[slot * 20 + j] = gb;
    __syncthreads();
    if (tid < 20) {
      double t = 0.0;
      for (int k = 0; k < kSlots; ++k) t += red[k * 20 + tid];
      if (t != 0.0) atomicAdd(h.ds_b0 + tid, (float)t);
    }
  }
  if (tid == 0 && blockIdx.x == 0 && d.trace != nullptr) { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); d.trace[30] = t; d.trace[29] = (unsigned long long)n_barrier; }
}

// ================================================================================================ weight gradients
// dW_g[k][n] += sum_rows act(x)[r][x_off + k] dz[r][z_off + n];  db_g[n] += sum_rows dz[r][z_off + n].  One CTA of 128 threads takes
// (problem, group, block of 8 k, row split): a thread owns one column n and 8 k accumulators; act(x) of the CTA's rows goes
// through shared memory (broadcast), dz is read coalesced from the buffers the dX chain left behind.
namespace {
constexpr int kDwThreads = 128;
constexpr int kDwRows = 64;                                   // rows staged per round
struct DwProb {
  const float* X; int ldx; int x_off0, x_stride;             // x column offset of group g = x_off0 + g * x_stride (tower 2 wraps to 0: see x_mod)
  int x_mod;                                                  // != 0: x offset = ((g * x_stride) % x_mod)
  int bn;                                                     // batch-norm set applied to X on load (relu(bn(.))), or -1: raw
  const float* dZ; int lddz; int z_stride;                    // dz column offset of group g = g * z_stride
  int K, N, groups;
  float* dW; int w_stride; float* db; int b_stride;
  int kblocks, first_task;
};
struct DwPlan { DwProb p[7]; int n_prob; int splits; int total; };
}  // namespace

__global__ void __launch_bounds__(kDwThreads) k_head2_dw(const __grid_constant__ Head2 h, const __grid_constant__ DwPlan plan, int B) {
  __shared__ __align__(16) float xsm[kDwRows * 8];
  const int tid = threadIdx.x;
  int task = blockIdx.x / plan.splits;
  const int split = blockIdx.x % plan.splits;
  int pi = 0;
  while (pi + 1 < plan.n_prob && task >= plan.p[pi + 1].first_task) ++pi;
  const DwProb& P = plan.p[pi];
  task -= P.first_task;
  const int g = task / P.kblocks, kb = task % P.kblocks;
  const int k0 = kb * 8, kn = min(8, P.K - k0);
  const int xo = (P.x_mod ? (g * P.x_stride) % P.x_mod : P.x_off0 + g * P.x_stride) + k0;
  const int zo = g * P.z_stride;
  const int rows_per = (B + plan.splits - 1) / plan.splits;
  const int r_begin = split * rows_per, r_end = min(B, r_begin + rows_per);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float sb = 0.f;
  const int n = tid;
  for (int r0 = r_begin; r0 < r_end; r0 += kDwRows) {
    const int nr = min(kDwRows, r_end - r0);
    __syncthreads();
    for (int i = tid; i < kDwRows * 8; i += kDwThreads) {
      const int r = i >> 3, kk = i & 7;
      float v = 0.f;
      if (r < nr && kk < kn) {
        v = P.X[(int64_t)(r0 + r) * P.ldx + xo + kk];
        if (P.bn >= 0) v = bn_act(v, bn_c(h.bn[P.bn], xo + kk));
      }
      xsm[i] = v;
    }
    __syncthreads();
    if (n < P.N) {
      const float* dz = P.dZ + (int64_t)r0 * P.lddz + zo + n;
#pragma unroll 4
      for (int r = 0; r < nr; ++r) {
        const float z = dz[(int64_t)r * P.lddz];
        const float4 a = ld4(xsm + r * 8), b = ld4(xsm + r * 8 + 4);
        acc[0] = fmaf(a.x, z, acc[0]); acc[1] = fmaf(a.y, z, acc[1]); acc[2] = fmaf(a.z, z, acc[2]); acc[3] = fmaf(a.w, z, acc[3]);
        acc[4] = fmaf(b.x, z, acc[4]); acc[5] = fmaf(b.y, z, acc[5]); acc[6] = fmaf(b.z, z, acc[6]); acc[7] = fmaf(b.w, z, acc[7]);
        sb += z;
      }
    }
  }
  if (n < P.N) {
    float* dW = P.dW + (int64_t)g * P.w_stride + (int64_t)k0 * P.N + n;
#pragma unroll
    for (int i = 0; i < 8; ++i) if (i < kn) atomicAdd(dW + (int64_t)i * P.N, acc[i]);
    if (kb == 0) atomicAdd(P.db + (int64_t)g * P.b_stride + n, sb);
  }
}

// ================================================================================================ host side
constexpr size_t kFwdSmem = (size_t)(kWBuf + kXS * kRC) * sizeof(float);
constexpr size_t kBwdSmem = (size_t)(kWBuf + kXS * kRC + 4096) * sizeof(float);
int head2_grid() {
  int dev = 0, sms = 0, coop = 0, occ_f = 0, occ_b = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return -1;
  if (cudaFuncSetAttribute(k_head2_fwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFwdSmem) != cudaSuccess) return -1;
  if (cudaFuncSetAttribute(k_head2_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBwdSmem) != cudaSuccess) return -1;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
  cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
  if (!coop) return -1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_f, k_head2_fwd, kT2, kFwdSmem) != cudaSuccess || occ_f < 1) return -1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_b, k_head2_bwd, kT2, kBwdSmem) != cudaSuccess || occ_b < 1) return -1;
  return sms;
}

int launch_head2_fwd(const Head2& h, const HeadDyn& d, int grid, const char* name, cudaStream_t st) {
  PAMREC_PROF(name, 1, st);
  if (d.B == 0 && d.world == 1) return 0;
  void* args[2] = {(void*)&h, (void*)&d};
  return cudaLaunchCooperativeKernel((const void*)k_head2_fwd, dim3(grid), dim3(kT2), args, kFwdSmem, st) == cudaSuccess ? 0 : -1;
}
int launch_head2_bwd(const Head2& h, const HeadDyn& d, int grid, cudaStream_t st) {
  PAMREC_PROF("head_bwd", 1, st);
  if (d.B == 0 && d.world == 1) return 0;
  void* args[2] = {(void*)&h, (void*)&d};
  return cudaLaunchCooperativeKernel((const void*)k_head2_bwd, dim3(grid), dim3(kT2), args, kBwdSmem, st) == cudaSuccess ? 0 : -1;
}
void launch_head2_dw(const Head2& h, int B, cudaStream_t st) {
  PAMREC_PROF("head_dw", 1, st);
  if (B == 0) return;
  DwPlan pl;
  memset(&pl, 0, sizeof pl);
  auto add = [&](const float* X, int ldx, int x_stride, int x_mod, int bn, const float* dZ, int lddz, int z_stride, int K, int N, int groups,
                 float* dW, int w_stride, float* db, int b_stride) {
    DwProb& p = pl.p[pl.n_prob++];
    p.X = X; p.ldx = ldx; p.x_off0 = 0; p.x_stride = x_stride; p.x_mod = x_mod; p.bn = bn; p.dZ = dZ; p.lddz = lddz; p.z_stride = z_stride;
    p.K = K; p.N = N; p.groups = groups; p.dW = dW; p.w_stride = w_stride; p.db = db; p.b_stride = b_stride;
    p.kblocks = (K + 7) / 8; p.first_task = pl.total;
    pl.total += groups * p.kblocks;
  };
  add(h.zt1, 192, 64, 0, BN_T1, h.d_logits, 3, 1, 64, 1, 3, h.dt_wo, 64, h.dt_bo, 1);                 // tower outputs
  add(h.zt0, 300, 100, 0, BN_T0, h.d_t1, 192, 64, 100, 64, 3, h.dt_w1, 6400, h.dt_b1, 64);           // towers layer 1
  add(h.u, 168, 84, 168, -1, h.d_t0, 300, 100, 84, 100, 3, h.dt_w0, 8400, h.dt_b0, 100);             // towers layer 0: inputs at 0, 84, 0
  add(h.ze0, 500, 100, 0, BN_E0, h.d_e1, 320, 64, 100, 64, 5, h.de_w1, 6400, h.de_b1, 64);           // experts layer 1
  add(h.zg0, 128, 64, 0, BN_G0, h.d_g1, 10, 5, 64, 5, 2, h.dg_w1, 320, h.dg_b1, 5);                  // gates layer 1
  add(h.new_long, kD, 0, 0, -1, h.d_e0, 500, 100, kD, 100, 5, h.de_w0, 4000, h.de_b0, 100);          // experts layer 0
  add(h.new_long, kD, 0, 0, -1, h.d_g0, 128, 64, kD, 64, 2, h.dg_w0, 2560, h.dg_b0, 64);             // gates layer 0
  pl.splits = (B + 255) / 256;
  if (pl.splits > 64) pl.splits = 64;
  k_head2_dw<<<pl.total * pl.splits, kDwThreads, 0, st>>>(h, pl, B);
}

}  // namespace pamrec
