// Attention on the tensor cores with warp-level MMAs (mma.sync.m16n8k8 TF32, error-compensated 3xTF32 split of mma.cuh):
//
//   S = Q K^T / sqrt(40),  P = softmax_j(mask_j ? S : -(2^32)+1),  y = P V + qin                      (pamrec.py:768-810)
//   backward: dQ = dS K,  dK = dS^T Q,  dV = P^T dY  with  dS = P o (dY V^T - D) / sqrt(40),  D_t = dY_t . (P V)_t
//
// Why m16n8k8 and not tcgen05 here: a sample is a 50 x 50 (T x T) problem.  A tcgen05 tile is 128 rows - two and a half samples of
// padding per sample at T = 50 (measured: a tcgen05 forward lost to the FFMA kernel, DESIGN.md section 4) - while a
// 16-row warp tile wastes 14 of 64 rows.  The FFMA kernels (kernels_encoder.cu) are bound by the latency of one thread's serial
// walk over the keys at 10 % occupancy; here a warp owns 16 query rows (or 16 key rows), scores live in accumulator fragments,
// and the probabilities feed the second product straight from registers: within a block of 8 keys the product's contraction
// index is permuted (fragment column t <-> key 2t, column t + 4 <-> key 2t + 1) so that the C fragment of S IS the A fragment
// of P - no shuffles, no shared-memory round trip.
//
// Only the LIVE keys of a sample are staged (compacted rows; a masked key's weight is exactly 0 as soon as the sample has one
// live key; a sample without any gets uniform weights like the reference) - at the bench's uniform history lengths half the MMAs.
// Backward = two passes like the FFMA kernel: pass A (warp = 16 queries) recomputes S, forms dP, dS and dQ; pass B (warp = 16
// keys) recomputes S^T = K Q^T against ALL queries, forms P^T and dS^T from the saved row statistics and accumulates dV = P^T dY,
// dK = dS^T Q.  Everything is warp-local: no atomics, sums in a fixed order.
#include <cstdlib>

#include "kernels.h"
#include "mma.cuh"

namespace pamrec {

namespace amma {

constexpr int kSt = 44;                    // shared-memory row stride (floats): conflict-free fragment loads (banks 12 g + t)
constexpr int kThreads = 128;              // 4 warps = 64 query (or key) rows per CTA; grid.y covers longer sequences

__device__ __forceinline__ void live_list(const int* __restrict__ mk, int T, int lane, int* __restrict__ lv, int* __restrict__ nl) {
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
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}
// A fragments (hi / lo) of 16 rows x 40 columns read from global memory: rows ra = r0 + g and rb = ra + 8 (zero beyond n_rows)
__device__ __forceinline__ void load_a_rows(const float* __restrict__ X, int64_t base_row, int ra, int rb, int n_rows, int t,
                                            uint32_t (&hi)[5][4], uint32_t (&lo)[5][4]) {
  const float* pa = X + (base_row + ra) * kD;
  const float* pb = X + (base_row + rb) * kD;
#pragma unroll
  for (int k0 = 0; k0 < 5; ++k0) {
    const int c = 8 * k0 + t;
    split_tf32(ra < n_rows ? pa[c] : 0.f, hi[k0][0], lo[k0][0]);
    split_tf32(rb < n_rows ? pb[c] : 0.f, hi[k0][1], lo[k0][1]);
    split_tf32(ra < n_rows ? pa[c + 4] : 0.f, hi[k0][2], lo[k0][2]);
    split_tf32(rb < n_rows ? pb[c + 4] : 0.f, hi[k0][3], lo[k0][3]);
  }
}
// c[4] += A[16 x 40] . R^T for the 8 rows n0 .. n0 + 7 of a shared-memory matrix R (row stride kSt): c[e] belongs to column n0 + 2t (+1)
__device__ __forceinline__ void mma_rows_t(float (&c)[4], const uint32_t (&ahi)[5][4], const uint32_t (&alo)[5][4],
                                           const float* __restrict__ R, int n0, int g, int t) {
  const float* r = R + (n0 + g) * kSt + t;
  // the three split terms run as three independent accumulation chains of 5 MMAs (one chain of 15 would serialise on the MMA
  // latency: a warp has only this tile in flight); small terms are added first
  float d1[4] = {0.f, 0.f, 0.f, 0.f}, d2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int k0 = 0; k0 < 5; ++k0) {
    uint32_t bh[2], bl[2];
    split_tf32(r[8 * k0], bh[0], bl[0]);
    split_tf32(r[8 * k0 + 4], bh[1], bl[1]);
    mma_tf32(d1, alo[k0], bh);
    mma_tf32(d2, ahi[k0], bl);
    mma_tf32(c, ahi[k0], bh);
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) c[e] += d1[e] + d2[e];
}
// o[5][4] += P[16 x 8] . R[8 x 40] where P is a C fragment reused as A fragment: fragment column t <-> row k0 + 2t of R, t + 4 <-> k0 + 2t + 1
__device__ __forceinline__ void mma_p_rows(float (&o)[5][4], const float (&p)[4], const float* __restrict__ R, int k0, int g, int t) {
  uint32_t ph[4], pl[4];
  split_tf32(p[0], ph[0], pl[0]);
  split_tf32(p[2], ph[1], pl[1]);
  split_tf32(p[1], ph[2], pl[2]);
  split_tf32(p[3], ph[3], pl[3]);
  const float* r0 = R + (k0 + 2 * t) * kSt + g;
#pragma unroll
  for (int nt = 0; nt < 5; ++nt) {
    uint32_t bh[2], bl[2];
    split_tf32(r0[8 * nt], bh[0], bl[0]);
    split_tf32(r0[kSt + 8 * nt], bh[1], bl[1]);
    mma_3xtf32(o[nt], ph, pl, bh, bl);
  }
}

// ------------------------------------------------------------------------------------------ forward
// shared memory: K | V (live rows, compacted, padded to a multiple of 8 with zeros) | mask | live list | count
__host__ __device__ inline size_t fwd_smem(int T) { const int Tp = (T + 7) & ~7, T4 = (T + 3) & ~3; return ((size_t)2 * Tp * kSt + 2 * T4 + 4) * 4; }

template <int NTM>
__global__ void __launch_bounds__(kThreads)
k_attn_fwd_mma(const float* __restrict__ Q, const float* __restrict__ K, const float* __restrict__ V, const float* __restrict__ QIN,
               const int* __restrict__ mask, float* __restrict__ Y, float* __restrict__ PV, float* __restrict__ ML, int T) {
  extern __shared__ __align__(16) float sm[];
  const int Tp = (T + 7) & ~7, T4 = (T + 3) & ~3;
  float* Ks = sm;
  float* Vs = Ks + Tp * kSt;
  int* mk = reinterpret_cast<int*>(Vs + Tp * kSt);
  int* lv = mk + T4;
  int* nlp = lv + T4;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int64_t base = (int64_t)b * T;
  for (int j = tid; j < T; j += kThreads) mk[j] = mask[base + j];
  __syncthreads();
  if (w == 0) live_list(mk, T, lane, lv, nlp);
  __syncthreads();
  int nl = *nlp;
  const bool uniform = nl == 0;              // no live key: every score is the padding constant, uniform weights over all T keys
  if (uniform) nl = T;
  const int nt_n = (nl + 7) >> 3;
  for (int i = tid; i < nt_n * 8 * 10; i += kThreads) {
    const int k = i / 10, c = i % 10;
    float4 kv = f4_zero(), vv = f4_zero();
    if (k < nl) {
      const int64_t gi = (base + (uniform ? k : lv[k])) * kD + 4 * c;
      kv = ld4(K + gi); vv = ld4(V + gi);
    }
    st4(Ks + k * kSt + 4 * c, kv);
    st4(Vs + k * kSt + 4 * c, vv);
  }
  __syncthreads();
  const int r0 = 64 * blockIdx.y + 16 * w;
  if (r0 >= T) return;
  const int g = lane >> 2, t = lane & 3;
  const int ra = r0 + g, rb = ra + 8;
  uint32_t qhi[5][4], qlo[5][4];
  load_a_rows(Q, base, ra, rb, T, t, qhi, qlo);
  const float rscale = 1.0f / sqrtf((float)kD);
  float c[NTM][4];
  float ma = -INFINITY, mb = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < NTM; ++nt) {
    if (nt < nt_n) {
      c[nt][0] = c[nt][1] = c[nt][2] = c[nt][3] = 0.f;
      mma_rows_t(c[nt], qhi, qlo, Ks, 8 * nt, g, t);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int key = 8 * nt + 2 * t + (e & 1);
        const float s = key < nl ? (uniform ? 0.f : c[nt][e] * rscale) : -INFINITY;
        c[nt][e] = s;
        if (e < 2) ma = fmaxf(ma, s); else mb = fmaxf(mb, s);
      }
    }
  }
  ma = quad_max(ma); mb = quad_max(mb);
  float la = 0.f, lb = 0.f;
  float o[5][4];
#pragma unroll
  for (int nt = 0; nt < 5; ++nt) o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.f;
#pragma unroll
  for (int nt = 0; nt < NTM; ++nt) {
    if (nt < nt_n) {
      c[nt][0] = expf(c[nt][0] - ma); c[nt][1] = expf(c[nt][1] - ma);
      c[nt][2] = expf(c[nt][2] - mb); c[nt][3] = expf(c[nt][3] - mb);
      la += c[nt][0] + c[nt][1];
      lb += c[nt][2] + c[nt][3];
      mma_p_rows(o, c[nt], Vs, 8 * nt, g, t);
    }
  }
  la = quad_sum(la); lb = quad_sum(lb);
  const float ia = 1.0f / la, ib = 1.0f / lb;
#pragma unroll
  for (int nt = 0; nt < 5; ++nt) {
    const int col = 8 * nt + 2 * t;
    if (ra < T) {
      const float2 r = *reinterpret_cast<const float2*>(QIN + (base + ra) * kD + col);
      *reinterpret_cast<float2*>(Y + (base + ra) * kD + col) = make_float2(fmaf(o[nt][0], ia, r.x), fmaf(o[nt][1], ia, r.y));
      *reinterpret_cast<float2*>(PV + (base + ra) * kD + col) = make_float2(o[nt][0] * ia, o[nt][1] * ia);
    }
    if (rb < T) {
      const float2 r = *reinterpret_cast<const float2*>(QIN + (base + rb) * kD + col);
      *reinterpret_cast<float2*>(Y + (base + rb) * kD + col) = make_float2(fmaf(o[nt][2], ib, r.x), fmaf(o[nt][3], ib, r.y));
      *reinterpret_cast<float2*>(PV + (base + rb) * kD + col) = make_float2(o[nt][2] * ib, o[nt][3] * ib);
    }
  }
  if (t == 0) {
    if (ra < T) { ML[2 * (base + ra)] = uniform ? kMaskNeg : ma; ML[2 * (base + ra) + 1] = la; }
    if (rb < T) { ML[2 * (base + rb)] = uniform ? kMaskNeg : mb; ML[2 * (base + rb) + 1] = lb; }
  }
}

// ------------------------------------------------------------------------------------------ backward
// shared memory: K | V (live rows, compacted, zero padded to a multiple of 16) | Q | dY (all T rows, zero padded to a multiple
// of 8) | m | 1 / l | D (per query, padded) | mask | live list | count
__host__ __device__ inline size_t bwd_smem(int T) {
  const int Tp8 = (T + 7) & ~7, Tp16 = (T + 15) & ~15, T4 = (T + 3) & ~3;
  return ((size_t)2 * Tp16 * kSt + 2 * Tp8 * kSt + 3 * Tp8 + 2 * T4 + 4) * 4;
}

__global__ void __launch_bounds__(kThreads, 3)      // 3 resident CTAs per SM: the most the registers allow without spills
k_attn_bwd_mma(const float* __restrict__ Q, const float* __restrict__ K, const float* __restrict__ V, const float* __restrict__ dY,
               const float* __restrict__ PV, const float* __restrict__ ML, const int* __restrict__ mask,
               float* __restrict__ dQ, float* __restrict__ dK, float* __restrict__ dV, int T) {
  extern __shared__ __align__(16) float sm[];
  const int Tp8 = (T + 7) & ~7, Tp16 = (T + 15) & ~15, T4 = (T + 3) & ~3;
  float* Ks = sm;
  float* Vs = Ks + Tp16 * kSt;
  float* Qs = Vs + Tp16 * kSt;
  float* Gs = Qs + Tp8 * kSt;
  float* rm = Gs + Tp8 * kSt;
  float* ril = rm + Tp8;
  float* rD = ril + Tp8;
  int* mk = reinterpret_cast<int*>(rD + Tp8);
  int* lv = mk + T4;
  int* nlp = lv + T4;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int64_t base = (int64_t)b * T;
  for (int j = tid; j < T; j += kThreads) mk[j] = mask[base + j];
  // Q, dY of every query row; D_t = dY_t . (P V)_t; row statistics.  Padding rows: zeros, statistics that give p = 0.
  for (int i = tid; i < Tp8 * 10; i += kThreads) {
    const int r = i / 10, c = i % 10;
    float4 q = f4_zero(), gy = f4_zero();
    if (r < T) { q = ld4(Q + (base + r) * kD + 4 * c); gy = ld4(dY + (base + r) * kD + 4 * c); }
    st4(Qs + r * kSt + 4 * c, q);
    st4(Gs + r * kSt + 4 * c, gy);
  }
  for (int r = tid; r < Tp8; r += kThreads) {
    float m = 0.f, il = 0.f, d = 0.f;
    if (r < T) {
      const int64_t tok = base + r;
#pragma unroll
      for (int i = 0; i < 10; ++i) {
        const float4 gy = ld4(dY + tok * kD + 4 * i), o = ld4(PV + tok * kD + 4 * i);
        d = fmaf(gy.x, o.x, d); d = fmaf(gy.y, o.y, d); d = fmaf(gy.z, o.z, d); d = fmaf(gy.w, o.w, d);
      }
      m = ML[2 * tok]; il = 1.0f / ML[2 * tok + 1];
    }
    rm[r] = m; ril[r] = il; rD[r] = d;
  }
  __syncthreads();
  if (w == 0) live_list(mk, T, lane, lv, nlp);
  __syncthreads();
  int nl = *nlp;
  const bool uniform = nl == 0;
  if (uniform) nl = T;
  const int nk16 = (nl + 15) >> 4, nt_n = (nl + 7) >> 3;
  for (int i = tid; i < nk16 * 16 * 10; i += kThreads) {
    const int k = i / 10, c = i % 10;
    float4 kv = f4_zero(), vv = f4_zero();
    if (k < nl) {
      const int64_t gi = (base + (uniform ? k : lv[k])) * kD + 4 * c;
      kv = ld4(K + gi); vv = ld4(V + gi);
    }
    st4(Ks + k * kSt + 4 * c, kv);
    st4(Vs + k * kSt + 4 * c, vv);
  }
  __syncthreads();
  const int g = lane >> 2, t = lane & 3;
  const float rscale = 1.0f / sqrtf((float)kD);
  const int r0 = 64 * blockIdx.y + 16 * w;
  // ---- pass A: the warp's 16 query rows against the live keys -> dQ
  if (r0 < T) {
    const int ra = r0 + g, rb = ra + 8;                                  // < Tp8 + 8: the statistics arrays are read below Tp8 only
    uint32_t qhi[5][4], qlo[5][4], ghi[5][4], glo[5][4];
    load_a_rows(Q, base, ra, rb, T, t, qhi, qlo);
    load_a_rows(dY, base, ra, rb, T, t, ghi, glo);
    const float m_a = ra < T ? rm[ra] : 0.f, m_b = rb < T ? rm[rb] : 0.f;
    const float il_a = ra < T ? ril[ra] : 0.f, il_b = rb < T ? ril[rb] : 0.f;
    const float D_a = ra < T ? rD[ra] : 0.f, D_b = rb < T ? rD[rb] : 0.f;
    float o[5][4];
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.f;
    if (!uniform) {                                                      // without a live key every score is a constant: dS = 0
#pragma unroll 1
      for (int nt = 0; nt < nt_n; ++nt) {
        float s[4] = {0.f, 0.f, 0.f, 0.f}, dp[4] = {0.f, 0.f, 0.f, 0.f};
        mma_rows_t(s, qhi, qlo, Ks, 8 * nt, g, t);
        mma_rows_t(dp, ghi, glo, Vs, 8 * nt, g, t);
        float ds[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = 8 * nt + 2 * t + (e & 1);
          const float p = key < nl ? expf(s[e] * rscale - (e < 2 ? m_a : m_b)) * (e < 2 ? il_a : il_b) : 0.f;
          ds[e] = p * (dp[e] - (e < 2 ? D_a : D_b)) * rscale;
        }
        mma_p_rows(o, ds, Ks, 8 * nt, g, t);
      }
    }
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const int col = 8 * nt + 2 * t;
      if (ra < T) *reinterpret_cast<float2*>(dQ + (base + ra) * kD + col) = make_float2(o[nt][0], o[nt][1]);
      if (rb < T) *reinterpret_cast<float2*>(dQ + (base + rb) * kD + col) = make_float2(o[nt][2], o[nt][3]);
    }
  }
  // ---- pass B: the warp's 16 (compacted) key rows against ALL queries -> dK, dV of those keys; masked keys get zeros
  // (a sample without live keys: "uniform", every key has p = 1 / T and dS = 0)
  const int k0 = 64 * blockIdx.y + 16 * w;                               // compacted key rows k0 .. k0 + 15
  if (k0 < nk16 * 16) {
    const int ka = k0 + g, kb = ka + 8;
    uint32_t khi[5][4], klo[5][4], vhi[5][4], vlo[5][4];
    {
      // A fragments of the warp's key rows from shared memory (rows beyond nl are zero)
      const float* pa = Ks + ka * kSt;
      const float* pb = Ks + kb * kSt;
      const float* va = Vs + ka * kSt;
      const float* vb = Vs + kb * kSt;
#pragma unroll
      for (int q0 = 0; q0 < 5; ++q0) {
        const int c = 8 * q0 + t;
        split_tf32(pa[c], khi[q0][0], klo[q0][0]); split_tf32(pb[c], khi[q0][1], klo[q0][1]);
        split_tf32(pa[c + 4], khi[q0][2], klo[q0][2]); split_tf32(pb[c + 4], khi[q0][3], klo[q0][3]);
        split_tf32(va[c], vhi[q0][0], vlo[q0][0]); split_tf32(vb[c], vhi[q0][1], vlo[q0][1]);
        split_tf32(va[c + 4], vhi[q0][2], vlo[q0][2]); split_tf32(vb[c + 4], vhi[q0][3], vlo[q0][3]);
      }
    }
    float ok[5][4], ov[5][4];
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) { ok[nt][0] = ok[nt][1] = ok[nt][2] = ok[nt][3] = 0.f; ov[nt][0] = ov[nt][1] = ov[nt][2] = ov[nt][3] = 0.f; }
    const bool live_a = ka < nl, live_b = kb < nl;
#pragma unroll 1
    for (int qt = 0; qt < Tp8 / 8; ++qt) {
      // S^T[key][query] and dP^T[key][query] for queries 8 qt .. 8 qt + 7 (fragment columns 2t, 2t + 1)
      float s[4] = {0.f, 0.f, 0.f, 0.f}, dp[4] = {0.f, 0.f, 0.f, 0.f};
      mma_rows_t(s, khi, klo, Qs, 8 * qt, g, t);
      mma_rows_t(dp, vhi, vlo, Gs, 8 * qt, g, t);
      float p[4], ds[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int q = 8 * qt + 2 * t + (e & 1);
        const bool live = e < 2 ? live_a : live_b;
        // padding queries carry il = 0; a sample without live keys: s = the padding constant = its own row maximum, p = 1 / l
        const float pe = live ? (uniform ? ril[q] : expf(s[e] * rscale - rm[q]) * ril[q]) : 0.f;
        p[e] = pe;
        ds[e] = uniform ? 0.f : pe * (dp[e] - rD[q]) * rscale;
      }
      mma_p_rows(ov, p, Gs, 8 * qt, g, t);
      mma_p_rows(ok, ds, Qs, 8 * qt, g, t);
    }
    // rows of the compacted list go back to their positions
    const int ja = live_a ? (uniform ? ka : lv[ka]) : -1, jb = live_b ? (uniform ? kb : lv[kb]) : -1;
#pragma unroll
    for (int nt = 0; nt < 5; ++nt) {
      const int col = 8 * nt + 2 * t;
      if (ja >= 0) {
        *reinterpret_cast<float2*>(dK + (base + ja) * kD + col) = make_float2(ok[nt][0], ok[nt][1]);
        *reinterpret_cast<float2*>(dV + (base + ja) * kD + col) = make_float2(ov[nt][0], ov[nt][1]);
      }
      if (jb >= 0) {
        *reinterpret_cast<float2*>(dK + (base + jb) * kD + col) = make_float2(ok[nt][2], ok[nt][3]);
        *reinterpret_cast<float2*>(dV + (base + jb) * kD + col) = make_float2(ov[nt][2], ov[nt][3]);
      }
    }
  }
  // masked keys (of a sample that has live ones): dK = dV = 0
  if (!uniform && blockIdx.y == 0) {
    for (int i = tid; i < T * 10; i += kThreads) {
      const int j = i / 10, c = i % 10;
      if (mk[j] == 0) { st4(dK + (base + j) * kD + 4 * c, f4_zero()); st4(dV + (base + j) * kD + 4 * c, f4_zero()); }
    }
  }
}

template <int NTM>
static void launch_fwd(const float* Q, const float* K, const float* V, const float* QIN, const int* mask, float* Y, float* PV, float* ML,
                       int B, int T, cudaStream_t st) {
  k_attn_fwd_mma<NTM><<<dim3(B, (T + 63) / 64), kThreads, fwd_smem(T), st>>>(Q, K, V, QIN, mask, Y, PV, ML, T);
}

}  // namespace amma

int init_attn_mma_kernels(int max_T) {
  cudaError_t e = cudaSuccess;
  auto set = [&](const void* fn, size_t bytes) {
    if (e == cudaSuccess && bytes > 48 * 1024) e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  };
  const size_t f = amma::fwd_smem(max_T), b = amma::bwd_smem(max_T);
  set((const void*)amma::k_attn_fwd_mma<7>, f);
  set((const void*)amma::k_attn_fwd_mma<13>, f);
  set((const void*)amma::k_attn_fwd_mma<25>, f);
  set((const void*)amma::k_attn_bwd_mma, b);
  return e == cudaSuccess ? 0 : -1;
}

void launch_attn_fwd_mma(const float* Q, const float* K, const float* V, const float* QIN, const int* mask, float* Y, float* PV, float* ML,
                         int B, int T, cudaStream_t st) {
  PAMREC_PROF("attn_fwd", 1, st);
  if (B == 0) return;
  if (T <= 56) amma::launch_fwd<7>(Q, K, V, QIN, mask, Y, PV, ML, B, T, st);
  else if (T <= 104) amma::launch_fwd<13>(Q, K, V, QIN, mask, Y, PV, ML, B, T, st);
  else amma::launch_fwd<25>(Q, K, V, QIN, mask, Y, PV, ML, B, T, st);      // up to 200 keys; the dispatch sends T <= 128 only
}

void launch_attn_bwd_mma(const float* Q, const float* K, const float* V, const float* dY, const float* PV, const float* ML,
                         const int* mask, float* dQ, float* dK, float* dV, int B, int T, cudaStream_t st) {
  PAMREC_PROF("attn_bwd", 1, st);
  if (B == 0) return;
  amma::k_attn_bwd_mma<<<dim3(B, (T + 63) / 64), amma::kThreads, amma::bwd_smem(T), st>>>(Q, K, V, dY, PV, ML, mask, dQ, dK, dV, T);
}

}  // namespace pamrec
